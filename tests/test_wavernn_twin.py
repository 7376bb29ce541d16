"""CPU tests of the WaveRNN oracle: the C twin (oracle/wavernn_twin.c) and the numpy post-processing
restatement are pinned against golden vectors generated from the LIVE reference
(oracle/make_golden_wavernn.py) - the integer samples must be identical."""
import json

import numpy as np
import pytest
import torch

import make_golden_pinned as mgp
import ref_init as ri
import wavernn_oracle as wo


@pytest.fixture(scope="module")
def twin():
    sd = ri.wavernn_state_dict(0, randomize_bn=True)
    return wo.Twin({k: v.numpy() for k, v in sd.items() if v.dtype == torch.float32})


@pytest.fixture(scope="module")
def gold(golden_dir):
    return np.load(golden_dir / "wavernn_seed0.npz")


def test_noise_stream_reproducible(gold):
    """the Exp(1) stream (two GRUCell constructions, then one exponential_ per step) regenerated on
    this host equals the stored head of the stream the reference consumed"""
    noise = ri.wavernn_noise(1234, 1, 128).numpy()
    assert np.array_equal(noise, gold["noise1_head"]), json.loads(str(gold["meta"]))


def test_twin_unbatched_prefix_matches_reference(twin, gold):
    """free-running twin == reference samples on the first 1500 draws (bit-exact integers)"""
    mel = gold["mel1"][0]
    aux, melup = twin.condition(mel)
    steps = 1500
    noise = ri.wavernn_noise(1234, 1, steps).numpy()
    idx = twin.generate(aux, melup, [0], steps, noise)
    assert np.array_equal(idx, gold["idx1"][:, :steps])


def test_twin_batched_folds_match_reference(twin, gold):
    """fold_with_overlap geometry + zero padding past the end + per-fold zero state: 6 folds"""
    mel = gold["mel2"][0]
    aux, melup = twin.condition(mel)
    nf, starts = wo.fold_geometry(30 * 200, 1000, 100)
    assert nf == 6 and gold["idx2"].shape == (6, 1200)
    steps = 400
    noise = ri.wavernn_noise(1234, nf, steps).numpy()
    idx = twin.generate(aux, melup, starts, steps, noise)
    assert np.array_equal(idx, gold["idx2"][:, :steps])


def test_postprocess_matches_reference(gold):
    w1 = wo.postprocess(gold["idx1"], 27, False, 8000, 400, ri.WAVERNN_HP)
    assert np.abs(w1 - gold["wav1"]).max() <= 1e-12
    w2 = wo.postprocess(gold["idx2"], 30, True, 1000, 100, ri.WAVERNN_HP)
    assert w2.shape == gold["wav2"].shape
    assert np.abs(w2 - gold["wav2"]).max() <= 1e-12


def test_scalar_math_accuracy():
    lib = wo.lib()
    xs = np.linspace(-20, 20, 4001, dtype=np.float32)
    e = np.array([lib.twin_expf(float(x)) for x in xs], dtype=np.float64)
    assert np.max(np.abs(e / np.exp(xs.astype(np.float64)) - 1)) < 4e-7
    s = np.array([lib.twin_sigmoidf(float(x)) for x in xs], dtype=np.float64)
    assert np.max(np.abs(s - 1 / (1 + np.exp(-xs.astype(np.float64))))) < 2e-7
    t = np.array([lib.twin_tanhf(float(x)) for x in xs], dtype=np.float64)
    assert np.max(np.abs(t - np.tanh(xs.astype(np.float64)))) < 3e-7
    us = np.exp(np.linspace(-16, 0, 2001)).astype(np.float32)
    lg = np.array([lib.twin_logf(float(u)) for u in us], dtype=np.float64)
    assert np.max(np.abs(lg - np.log(us.astype(np.float64)))) < 2e-6


def test_builtin_noise_is_exp1():
    lib = wo.lib()
    q = np.array([lib.twin_noise(7, s, 3, c) for s in range(40) for c in range(512)])
    assert q.min() > 0 and abs(q.mean() - 1.0) < 0.03 and abs(q.var() - 1.0) < 0.08


def test_ref_init_wavernn_bit_identical_to_reference_constructor(golden_dir):
    """names, dtypes, shapes and bits of the state dict == the reference constructor's (digest stored by
    oracle/make_golden_pinned.py)"""
    pinned = json.loads((golden_dir / "reference_pinned.json").read_text())
    sd = ri.wavernn_state_dict(4, randomize_bn=False)
    assert mgp.state_dict_digest(sd) == pinned["state_dicts"]["wavernn_seed4"]


def test_three_term_fp16_split_is_fp32_equivalent():
    """Arithmetic contract of the tensor-core recurrent GEMMs (csrc/tacotron_tc.cu): every product is computed as
    hi(a)hi(w) + lo(a)hi(w) + hi(a)lo(w) with hi = fp16(v), lo = fp16(v - hi), weights pre-scaled by a power of two,
    FP32 accumulation.  Emulated here in numpy on a K = 2048 dot product (the decoder LSTM shape): the split's error
    against float64 is of the order of a plain FP32 dot product's and ~1000x below a plain fp16-operand product's."""
    rng = np.random.default_rng(0)
    K, N = 2048, 512
    a = rng.standard_normal((8, K)).astype(np.float32)                      # activations O(1)
    w = (rng.uniform(-1, 1, (N, K)) / 32).astype(np.float32)                 # LSTM init scale 1/sqrt(1024)
    exact = a.astype(np.float64) @ w.astype(np.float64).T
    scale = np.float32(2.0 ** (12 - np.frexp(np.abs(w).max())[1]))           # max |w| * scale in [2^11, 2^12)
    ws = w * scale

    def hi(v):
        return v.astype(np.float16).astype(np.float32)

    def lo(v):
        return (v - hi(v)).astype(np.float16).astype(np.float32)

    split = (hi(a) @ hi(ws).T + lo(a) @ hi(ws).T + hi(a) @ lo(ws).T) / scale  # float32 matmuls = fp32 accumulation
    plain32 = a @ w.T
    plain16 = hi(a) @ hi(w).T
    ref = np.abs(exact).max()
    e_split, e32, e16 = (np.abs(x - exact).max() / ref for x in (split, plain32, plain16))
    assert e_split < 4 * max(e32, 1e-7), (e_split, e32)
    assert e_split < e16 / 200, (e_split, e16)
    assert e_split < 5e-6
