"""CPU tests: the oracle restatements and the seeded weights of synth_weights/ref_init.py are pinned against the
committed golden vectors that oracle/make_golden.py and oracle/make_golden_pinned.py produced from the LIVE reference."""
import json
import os

import numpy as np
import pytest
import torch

import gan_oracle as go
import make_golden_pinned as mgp
import ref_init as ri


@pytest.fixture(scope="module")
def pinned(golden_dir):
    return json.loads((golden_dir / "reference_pinned.json").read_text())


def test_hifigan_oracle_matches_golden(golden_dir):
    z = np.load(golden_dir / "hifigan_seed0.npz")
    sd = ri.hifigan_state_dict(ri.HIFIGAN_CONFIG_16K, 0)
    with torch.no_grad():
        wav = go.hifigan_forward(sd, ri.HIFIGAN_CONFIG_16K, torch.from_numpy(z["mel_small"]))
    e = go.rel_errors(wav, torch.from_numpy(z["wav_small"]))
    # same torch build -> bit-identical; other CPU capability / thread count -> last-ulp noise only
    assert e["max_rel"] < 1e-5 and e["rms_rel"] < 1e-5, (e, json.loads(str(z["meta"])))


def test_hifigan_oracle_matches_golden_full_length(golden_dir):
    z = np.load(golden_dir / "hifigan_seed0.npz")
    sd = ri.hifigan_state_dict(ri.HIFIGAN_CONFIG_16K, 0)
    mel = torch.rand(32, 80, 256, generator=torch.Generator().manual_seed(2)) * 8 - 4
    with torch.no_grad():
        wav = go.hifigan_forward(sd, ri.HIFIGAN_CONFIG_16K, mel[[int(i) for i in z["full_pick"]]])
    e = go.rel_errors(wav, torch.from_numpy(z["wav_full"]))
    assert e["max_rel"] < 1e-5, e


def test_fregan_oracle_matches_golden(golden_dir):
    z = np.load(golden_dir / "fregan_seed0.npz")
    sd = ri.fregan_state_dict(ri.FREGAN_CONFIG, 0)
    with torch.no_grad():
        wav = go.fregan_forward(sd, ri.FREGAN_CONFIG, torch.from_numpy(z["mel"]))
    e = go.rel_errors(wav, torch.from_numpy(z["wav"]))
    assert e["max_rel"] < 1e-5, e


def test_work_figures_match_survey():
    w = go.hifigan_work(ri.HIFIGAN_CONFIG_16K, 256)
    assert w["macs"] == 45_068_779_520          # SURVEY.md appendix A.1
    assert w["params"] == 12_975_745
    assert w["act_elems"] == 168_433_664
    assert w["samples"] == 51_200


def test_fold_weight_norm_identity():
    v = torch.randn(8, 4, 3)
    g = v.reshape(8, -1).norm(dim=1).reshape(8, 1, 1) * 2.0
    out = go.fold_weight_norm({"c.weight_g": g, "c.weight_v": v, "c.bias": torch.zeros(8)})
    assert torch.allclose(out["c.weight"], 2.0 * v, rtol=1e-6, atol=1e-7)


def test_ref_init_bit_identical_to_reference_constructors(pinned):
    """state dicts of `torch.manual_seed(s); Generator(h)` / `FreGAN(h)` (eval, weight norm removed): names, dtypes,
    shapes and bits equal the reference's (stored digests); the restated configs equal the reference's JSON configs"""
    sds = pinned["state_dicts"]
    assert mgp.state_dict_digest(ri.hifigan_state_dict(ri.HIFIGAN_CONFIG_16K, 5)) == sds["hifigan_seed5"]
    assert mgp.state_dict_digest(ri.fregan_state_dict(ri.FREGAN_CONFIG, 6)) == sds["fregan_seed6"]
    assert ri.HIFIGAN_CONFIG_16K == pinned["configs"]["hifigan"]
    assert ri.FREGAN_CONFIG == pinned["configs"]["fregan"]


def test_gan_oracles_bit_identical_to_reference_forward(pinned, golden_dir):
    """the oracle forwards on the reference's own seed-1 weights (bit-identical, stored digests) == the stored reference
    forwards up to the last-ulp noise of the CPU convolutions, which depends on the CPU capability and thread count: bit for
    bit with those of the recording (meta), 1.4e-6 max_rel with AVX2 or with one thread"""
    z = np.load(golden_dir / "reference_pinned.npz")
    x = torch.rand(2, 80, 24, generator=torch.Generator().manual_seed(3)) * 8 - 4
    g = ri.hifigan_state_dict(ri.HIFIGAN_CONFIG_16K, 1)
    f = ri.fregan_state_dict(ri.FREGAN_CONFIG, 1)
    assert mgp.state_dict_digest(g) == pinned["state_dicts"]["hifigan_seed1"]
    assert mgp.state_dict_digest(f) == pinned["state_dicts"]["fregan_seed1"]
    with torch.no_grad():
        for got, key in ((go.hifigan_forward(g, ri.HIFIGAN_CONFIG_16K, x), "hifigan_seed1_wav"),
                         (go.fregan_forward(f, ri.FREGAN_CONFIG, x), "fregan_seed1_wav")):
            e = go.rel_errors(got, torch.from_numpy(z[key]))
            assert e["max_rel"] < 1e-5 and e["rms_rel"] < 1e-5, (key, e, pinned["meta"])


def _unpack_masks(z, name, B, Tc):
    enc = np.unpackbits(z[f"{name}_enc_masks"], axis=-1).astype(bool)
    dec = np.unpackbits(z[f"{name}_dec_masks"], axis=-1).astype(bool)
    return [torch.from_numpy(m) for m in enc] + [torch.from_numpy(m) for m in dec]


@pytest.mark.parametrize("name", ["a", "b"])
def test_tacotron_oracle_matches_golden(golden_dir, name):
    """Tacotron.generate restatement with the captured PreNet dropout masks injected"""
    import tacotron_oracle as to

    z = np.load(golden_dir / "tacotron_seed0.npz")
    sd = ri.tacotron_state_dict(0, r=2, randomize_bn=True)
    chars, emb = torch.from_numpy(z[f"{name}_chars"]), torch.from_numpy(z[f"{name}_emb"])
    steps, style, mst, r = [int(v) for v in z[f"{name}_cfg"]]
    masks = _unpack_masks(z, name, *chars.shape)
    mel, linear, attn = to.generate(sd, chars, emb, steps, style, mst, masks, r=r)
    for got, key in ((mel, "mel"), (linear, "linear"), (attn, "attn")):
        ref = torch.from_numpy(z[f"{name}_{key}"])
        assert got.shape == ref.shape
        assert float((got - ref).abs().max() / ref.abs().max()) < 2e-5, key


def test_ref_init_tacotron_bit_identical(pinned):
    sd = ri.tacotron_state_dict(2, r=1, randomize_bn=False)
    assert mgp.state_dict_digest(sd) == pinned["state_dicts"]["tacotron_seed2"]


@pytest.mark.parametrize("name", ["a", "b"])
def test_encoder_oracle_matches_golden(golden_dir, name):
    """SpeakerEncoder.forward restatement vs the live-reference golden (model.py:41-61)"""
    import encoder_oracle as eo

    z = np.load(golden_dir / "encoder_seed0.npz")
    sd = ri.encoder_state_dict(0)
    got = eo.embed_frames(sd, torch.from_numpy(z[f"{name}_frames"])).numpy()
    assert np.abs(got - z[f"{name}_embeds"]).max() < 1e-6
    if name == "a":
        utt = eo.embed_utterance_partials(sd, torch.from_numpy(z["a_frames"]))
        assert np.abs(utt - z["a_utterance"]).max() < 1e-6
        assert abs(float(np.linalg.norm(utt)) - 1.0) < 1e-6


def test_ref_init_encoder_bit_identical(pinned):
    assert mgp.state_dict_digest(ri.encoder_state_dict(3)) == pinned["state_dicts"]["encoder_seed3"]


def test_encoder_partial_slices_match_reference_rule(pinned):
    """compute_partial_slices (encoder/inference.py:66-125): known cases incl. the coverage rule"""
    from mockingbird_b200.encoder.inference import compute_partial_slices

    w, m = compute_partial_slices(16000 * 3)  # 3 s: 301 frames, step 80
    assert [s.start for s in m] == [0, 80, 160] and all(s.stop - s.start == 160 for s in m)
    assert w[1] == slice(80 * 160, 240 * 160)
    w, m = compute_partial_slices(1000)  # shorter than one partial: always one slice
    assert len(m) == 1 and m[0] == slice(0, 160)
    w, m = compute_partial_slices(16000 * 3, min_pad_coverage=1.0)
    assert [s.start for s in m] == [0, 80]
    for case in pinned["partial_slices"]:
        w, m = compute_partial_slices(case["n"], **case["kw"])
        assert [mgp.slice_bounds(s) for s in w] == case["wav"] and [mgp.slice_bounds(s) for s in m] == case["mel"], case


def test_melspec_oracle_stft_matches_torch_and_mel_basis_matches_transformers():
    """The mel front-end oracle cannot be pinned to the reference (librosa is absent and unpinned there); its two
    halves are cross-checked against independent implementations of the same published algorithms instead."""
    import melspec_oracle as mo

    rng = np.random.default_rng(0)
    y = (rng.standard_normal(5000) * 0.1).astype(np.float32)
    for n_fft, hop, mode in ((400, 160, "reflect"), (1024, 256, "constant"), (1024, 256, "reflect")):
        D = mo.stft(y, n_fft, hop, n_fft, mode)
        T = torch.stft(torch.from_numpy(y).double(), n_fft, hop, n_fft,
                       window=torch.hann_window(n_fft, periodic=True, dtype=torch.float64), center=True, pad_mode=mode,
                       return_complex=True).numpy()
        assert D.shape == T.shape == (1 + n_fft // 2, 1 + len(y) // hop)
        assert np.abs(D - T).max() < 1e-10
    # transformers.audio_utils.mel_filter_bank is an independent implementation of librosa.filters.mel; it runs in a
    # fresh interpreter because the reference-import stubs of this test module shadow optional audio packages
    import subprocess
    import sys

    code = ("import numpy as np, sys\n"
            "from transformers.audio_utils import mel_filter_bank as m\n"
            "np.savez(sys.argv[1], a=m(201, 40, 0.0, 8000.0, 16000, norm='slaney', mel_scale='slaney').T,"
            " b=m(513, 80, 55.0, 7600.0, 16000, norm='slaney', mel_scale='slaney').T)\n")
    import tempfile

    with tempfile.TemporaryDirectory() as d:
        r = subprocess.run([sys.executable, "-c", code, d + "/mel.npz"], capture_output=True, text=True, timeout=300)
        if r.returncode != 0:  # pragma: no cover
            pytest.skip("transformers.audio_utils not usable: " + r.stderr[-200:])
        z = np.load(d + "/mel.npz")
        for key, (sr, n_fft, n_mels, fmin, fmax) in (("a", (16000, 400, 40, 0.0, 8000.0)), ("b", (16000, 1024, 80, 55.0, 7600.0))):
            ours = mo.mel_basis(sr, n_fft, n_mels, fmin, fmax)
            theirs = z[key]
            assert ours.shape == theirs.shape
            assert np.abs(ours - theirs).max() < 1e-6 * max(1.0, float(np.abs(theirs).max()))


def test_deepmind_oracle_matches_reference(golden_dir, pinned):
    """N3: ref_init reproduces the constructor of the UNMODIFIED deepmind_version.py (run behind the harness stubs when the
    digest was stored) bit for bit; the torch restatement reproduces the reference's integer coarse / fine samples and
    combined output (stored by oracle/make_golden_deepmind.py)"""
    import deepmind_oracle as do

    fresh = ri.deepmind_state_dict(0, bias_scale=0.0)
    assert mgp.state_dict_digest(fresh) == pinned["state_dicts"]["deepmind_seed0"]
    sd = ri.deepmind_state_dict(0)
    torch.manual_seed(1234)
    out, c, f = do.generate(sd, 600)
    z = np.load(golden_dir / "deepmind_seed0.npz")
    assert np.array_equal(z["coarse"][:600], c) and np.array_equal(z["fine"][:600], f)
    assert np.array_equal(z["output"][:600], out)


def test_deepmind_oracle_matches_golden(golden_dir):
    """runs everywhere (no reference tree needed): the restatement reproduces the committed reference samples"""
    import deepmind_oracle as do

    z = np.load(golden_dir / "deepmind_seed0.npz")
    sd = ri.deepmind_state_dict(0)
    torch.manual_seed(1234)
    out, c, f = do.generate(sd, 1000)
    assert np.array_equal(c, z["coarse"][:1000]) and np.array_equal(f, z["fine"][:1000])
    assert np.array_equal(out, z["output"][:1000]) and out.min() >= -2 ** 15 and out.max() < 2 ** 15
