"""Oracle for monotonic_align.maximum_path (TEST INFRASTRUCTURE; SURVEY.md 8f row N4).

  maximum_path_numpy   plain restatement of monotonic_align/core.pyx:7-42 (`maximum_path_each`) and of the wrapper
                       monotonic_align/__init__.py:6-19 (float32 DP in place, int32 path)
  reference_core()     the reference's OWN core.pyx compiled by oracle/build_oracle.build_ref() into oracle/_ref (the module's
                       init symbol is PyInit_core, so it is loaded under the name "core")
  random_case()        the seeded inputs of tests/test_monotonic.py
oracle/make_golden_pinned.py stores the compiled reference's paths and values on those inputs; tests/test_monotonic.py checks
restatement == compiled reference (bit-identical values and paths) and CUDA == both."""
from __future__ import annotations

import importlib.machinery
import importlib.util

import numpy as np

import build_oracle


def reference_core():
    so = build_oracle.ref_so() or build_oracle.build_ref()
    if so is None:
        return None
    loader = importlib.machinery.ExtensionFileLoader("core", str(so))
    spec = importlib.util.spec_from_loader("core", loader)
    mod = importlib.util.module_from_spec(spec)
    loader.exec_module(mod)
    return mod


def maximum_path_each(path: np.ndarray, value: np.ndarray, t_y: int, t_x: int, max_neg_val: float = -1e9) -> None:
    """core.pyx:7-37, in place on float32 `value` [T_y, T_x] and int32 `path`"""
    neg = np.float32(max_neg_val)
    index = t_x - 1
    for y in range(t_y):
        for x in range(max(0, t_x + y - t_y), min(t_x, y + 1)):
            v_cur = neg if x == y else value[y - 1, x]
            if x == 0:
                v_prev = np.float32(0.0) if y == 0 else neg
            else:
                v_prev = value[y - 1, x - 1]
            value[y, x] = np.float32(value[y, x] + max(v_prev, v_cur))
    for y in range(t_y - 1, -1, -1):
        path[y, index] = 1
        if index != 0 and (index == y or value[y - 1, index] < value[y - 1, index - 1]):
            index -= 1


def maximum_path_numpy(neg_cent: np.ndarray, t_ys: np.ndarray, t_xs: np.ndarray):
    """-> (paths int32 [b, T_y, T_x], values float32 after the in-place DP)"""
    values = np.ascontiguousarray(neg_cent, dtype=np.float32).copy()
    paths = np.zeros(values.shape, dtype=np.int32)
    for b in range(values.shape[0]):
        maximum_path_each(paths[b], values[b], int(t_ys[b]), int(t_xs[b]))
    return paths, values


def random_case(seed: int, b: int, ty: int, tx: int):
    """-> (neg_cent float32 [b, ty, tx], t_ys int32 [b], t_xs int32 [b]); row 0 spans the whole grid"""
    rng = np.random.RandomState(seed)
    v = (rng.randn(b, ty, tx) * 3).astype(np.float32)
    t_ys = rng.randint(max(1, ty // 2), ty + 1, size=b).astype(np.int32)
    t_xs = np.minimum(rng.randint(1, tx + 1, size=b), t_ys).astype(np.int32)  # a monotonic path needs t_x <= t_y
    t_ys[0], t_xs[0] = ty, min(tx, ty)
    return v, t_ys, t_xs
