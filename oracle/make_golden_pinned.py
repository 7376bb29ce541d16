"""Golden fixtures that pin synth_weights/ref_init.py and the oracle restatements to the LIVE reference, so that the tests
which check them need no reference tree (TEST INFRASTRUCTURE; needs the reference, see ref_harness.REFERENCE_ROOT).

    CUDA_VISIBLE_DEVICES="" python oracle/make_golden_pinned.py

  reference_pinned.json  digests (SHA-256 of every name, dtype, shape and the bytes) of the reference constructors' state
                         dicts: HiFi-GAN seed 5 and seed 1, Fre-GAN seed 6 and seed 1 (eval, weight norm removed),
                         Tacotron seed 2, SpeakerEncoder seed 3, fatchord WaveRNN seed 4, DeepMind WaveRNN seed 0; the two
                         GAN configs (the keys ref_init restates); encoder compute_partial_slices on a grid of lengths and options; text_to_sequence ids
  reference_pinned.npz   the reference HiFi-GAN / Fre-GAN forward with the seed-1 weights on rand(2,80,24;seed 3)*8-4; the
                         reference's own compiled monotonic_align core (oracle/build_oracle.build_ref) on the cases of
                         tests/test_monotonic.py: bit-packed paths and digests of the in-place DP values
"""
from __future__ import annotations

import hashlib
import json
import sys
from pathlib import Path

import numpy as np

HERE = Path(__file__).resolve().parent
GOLDEN = HERE.parent / "tests" / "golden"
JSON_PATH = GOLDEN / "reference_pinned.json"
NPZ_PATH = GOLDEN / "reference_pinned.npz"

# (seed, shapes) of the monotonic_align cases: tests/test_monotonic.py parametrizes over the same lists
MONOTONIC_CASES = {1: [(3, 37, 11), (2, 1, 1), (4, 64, 64), (2, 300, 75)],
                   2: [(3, 37, 11), (2, 1, 1), (4, 64, 64), (16, 1000, 200), (2, 300, 75)]}
PARTIAL_SLICE_LENGTHS = [1000, 25601, 48000, 51199, 160000]
PARTIAL_SLICE_OPTIONS = [{}, {"overlap": 0.25}, {"rate": 1.3}, {"min_pad_coverage": 0.5}]
TEXTS = ["ni3 hao3 shi4 jie4", "Mixed CASE,  spaces!", "~_skip~"]


def array_digest(a: np.ndarray) -> str:
    a = np.ascontiguousarray(a)
    h = hashlib.sha256(f"{a.dtype.str}{a.shape}".encode())
    h.update(a.tobytes())
    return h.hexdigest()


def state_dict_digest(sd) -> str:
    """one digest of every (name, dtype, shape, bits) of a state dict, independent of the key order"""
    h = hashlib.sha256()
    for k in sorted(sd):
        h.update(k.encode())
        h.update(array_digest(sd[k].detach().cpu().numpy()).encode())
    return h.hexdigest()


def slice_bounds(s: slice) -> list:
    return [None if v is None else int(v) for v in (s.start, s.stop, s.step)]


def monotonic_key(seed: int, shape) -> str:
    return f"monotonic_seed{seed}_" + "x".join(str(s) for s in shape)


def _generate():
    import torch

    import monotonic_oracle as mo
    import ref_harness as rh
    import ref_init as ri
    from make_golden import meta

    rh.install()
    rh.hide_cuda()
    out = {"meta": json.loads(meta())}
    arrays = {}
    sds = out["state_dicts"] = {}
    sds["hifigan_seed5"] = state_dict_digest(rh.build_hifigan(seed=5).state_dict())
    sds["fregan_seed6"] = state_dict_digest(rh.build_fregan(seed=6).state_dict())
    sds["tacotron_seed2"] = state_dict_digest(rh.build_tacotron(seed=2).state_dict())
    sds["encoder_seed3"] = state_dict_digest(rh.build_encoder(seed=3).state_dict())
    sds["wavernn_seed4"] = state_dict_digest(rh.build_wavernn(seed=4).state_dict())
    out["configs"] = {"hifigan": {k: rh.hifigan_config()[k] for k in ri.HIFIGAN_CONFIG_16K},
                      "fregan": {k: rh.fregan_config()[k] for k in ri.FREGAN_CONFIG}}

    x = torch.rand(2, 80, 24, generator=torch.Generator().manual_seed(3)) * 8 - 4
    g = rh.build_hifigan(seed=1)
    f = rh.build_fregan(seed=1)
    sds["hifigan_seed1"] = state_dict_digest(g.state_dict())
    sds["fregan_seed1"] = state_dict_digest(f.state_dict())
    with torch.no_grad():
        arrays["hifigan_seed1_wav"] = g(x).numpy()
        arrays["fregan_seed1_wav"] = f(x).numpy()

    from models.encoder import inference as ref_inf
    from models.synthesizer.utils.text import text_to_sequence

    out["partial_slices"] = [
        {"n": n, "kw": kw, "wav": [slice_bounds(s) for s in w], "mel": [slice_bounds(s) for s in m]}
        for n in PARTIAL_SLICE_LENGTHS for kw in PARTIAL_SLICE_OPTIONS
        for w, m in [ref_inf.compute_partial_slices(n, **kw)]]
    out["text_to_sequence"] = [{"text": t, "ids": text_to_sequence(t, ["basic_cleaners"])} for t in TEXTS]

    W = rh.load_deepmind()
    torch.manual_seed(0)
    sds["deepmind_seed0"] = state_dict_digest(W().state_dict())

    core = mo.reference_core()  # builds oracle/_ref on first use
    for seed, shapes in MONOTONIC_CASES.items():
        for shape in shapes:
            v, t_ys, t_xs = mo.random_case(seed, *shape)
            p, vv = np.zeros(v.shape, np.int32), v.copy()
            core.maximum_path_c(p, vv, t_ys, t_xs)
            assert set(np.unique(p)) <= {0, 1}
            key = monotonic_key(seed, shape)
            arrays[key + "_path"] = np.packbits(p.astype(np.uint8).ravel())
            out.setdefault("monotonic_values", {})[key] = array_digest(vv)

    JSON_PATH.write_text(json.dumps(out, indent=1, sort_keys=True) + "\n")
    np.savez_compressed(NPZ_PATH, **arrays)
    for p in (JSON_PATH, NPZ_PATH):
        print(p.name, p.stat().st_size)


if __name__ == "__main__":
    import os

    os.environ.setdefault("CUDA_VISIBLE_DEVICES", "")
    sys.path.insert(0, str(HERE))
    sys.path.insert(0, str(HERE.parent / "synth_weights"))
    _generate()
