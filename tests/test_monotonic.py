"""monotonic_align.maximum_path (SURVEY.md 8f row N4): numpy restatement == the reference's own compiled core.pyx == the CUDA
wavefront DP.  The compiled reference's paths and DP values on these cases are stored by oracle/make_golden_pinned.py."""
import json

import numpy as np
import pytest
import torch

import make_golden_pinned as mgp
import monotonic_oracle as mo


@pytest.fixture(scope="module")
def golden(golden_dir):
    return json.loads((golden_dir / "reference_pinned.json").read_text()), np.load(golden_dir / "reference_pinned.npz")


def _reference_path(golden, seed, shape):
    bits = golden[1][mgp.monotonic_key(seed, shape) + "_path"]
    return np.unpackbits(bits, count=int(np.prod(shape))).reshape(shape).astype(np.int32)


@pytest.mark.parametrize("shape", mgp.MONOTONIC_CASES[1])
def test_restatement_equals_compiled_reference(shape, golden):
    v, t_ys, t_xs = mo.random_case(1, *shape)
    p, vv = mo.maximum_path_numpy(v, t_ys, t_xs)
    assert np.array_equal(p, _reference_path(golden, 1, shape))
    assert mgp.array_digest(vv) == golden[0]["monotonic_values"][mgp.monotonic_key(1, shape)]
    assert np.array_equal(p.sum(axis=(1, 2)), t_ys)  # one cell per frame


@pytest.mark.gpu
@pytest.mark.parametrize("shape", mgp.MONOTONIC_CASES[2])
def test_cuda_equals_reference(shape, golden):
    from mockingbird_b200.monotonic_align import maximum_path

    v, t_ys, t_xs = mo.random_case(2, *shape)
    b, ty, tx = shape
    mask = np.zeros((b, ty, tx), np.float32)
    for i in range(b):
        mask[i, : t_ys[i], : t_xs[i]] = 1
    got = maximum_path(torch.from_numpy(v).cuda(), torch.from_numpy(mask).cuda())
    assert got.dtype == torch.float32 and got.shape == (b, ty, tx)
    assert np.array_equal(got.cpu().numpy().astype(np.int32), _reference_path(golden, 2, shape))
    # size-independent properties: exactly one cell per valid frame, monotone non-decreasing column, ends at the corners
    g = got.cpu().numpy()
    for i in range(b):
        cols = g[i, : t_ys[i]].argmax(axis=1)
        assert g[i].sum() == t_ys[i] and cols[0] == 0 and cols[-1] == t_xs[i] - 1
        assert np.all(np.diff(cols) >= 0) and np.all(np.diff(cols) <= 1)
