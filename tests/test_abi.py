"""CPU tests: the C-ABI library loads and exports every symbol include/mockingbird_b200.h declares;
handle creation / plan building / error paths work without a GPU (no compute calls)."""
import ctypes as C
import json
import re
from pathlib import Path

import pytest

from mockingbird_b200 import _lib

ROOT = Path(__file__).resolve().parent.parent


def declared_symbols():
    text = (ROOT / "include" / "mockingbird_b200.h").read_text()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(mb_[a-z0-9_]+)\s*\(", text)))


def test_header_symbols_exported_and_bound():
    lib = _lib.lib()
    syms = declared_symbols()
    assert len(syms) >= 20
    for s in syms:
        assert hasattr(lib, s), f"{s} declared in the header but not exported"
        assert s in _lib.SIGNATURES, f"{s} has no ctypes signature"
    assert lib.mb_version().startswith(b"mockingbird_b200")


def _hifigan_cfg(precision=_lib.MB_PREC_FP32):
    from mockingbird_b200.vocoder.hifigan.models import DEFAULT_CONFIG_16K as h

    cfg = _lib.GanConfig()
    cfg.kind = _lib.MB_GAN_HIFIGAN
    cfg.num_mels = 80
    cfg.upsample_initial_channel = h["upsample_initial_channel"]
    cfg.num_upsamples = 4
    for i in range(4):
        cfg.upsample_rates[i] = h["upsample_rates"][i]
        cfg.upsample_kernel_sizes[i] = h["upsample_kernel_sizes"][i]
    cfg.num_kernels = 3
    cfg.num_dilations = 3
    for j in range(3):
        cfg.resblock_kernel_sizes[j] = h["resblock_kernel_sizes"][j]
        for m in range(3):
            cfg.resblock_dilation_sizes[j][m] = h["resblock_dilation_sizes"][j][m]
    cfg.resblock_type = 1
    cfg.fregan_top_k = 4
    cfg.precision = precision
    return cfg


@pytest.mark.parametrize("precision", [_lib.MB_PREC_FP32, _lib.MB_PREC_F16TC])
def test_gan_plan_shape(precision):
    lib = _lib.lib()
    h = C.c_void_p()
    cfg = _hifigan_cfg(precision)
    _lib.check(lib.mb_gan_create(C.byref(cfg), C.byref(h)))
    try:
        assert lib.mb_gan_hop(h) == 200
        # conv_pre + 4 ups + 72 resblock convs + conv_post (SURVEY.md appendix A.1)
        assert lib.mb_gan_num_layers(h) == 78
        buf = C.create_string_buffer(256)
        _lib.check(lib.mb_gan_layer_info(h, 0, buf, 256))
        assert b"conv_pre" in buf.value and b"cin=80" in buf.value
        assert lib.mb_gan_arena_bytes(h) >= 12_975_745 * 4
        assert lib.mb_gan_workspace_bytes(h, 2, 16) > 0
        # forward before weights are set must fail loudly, not compute
        rc = lib.mb_gan_forward(h, C.c_void_p(256), None, 1, 8, C.c_void_p(256), C.c_void_p(256), 1 << 30, None)
        assert rc == 2 and b"finalized" in lib.mb_last_error()
    finally:
        lib.mb_gan_destroy(h)


def test_gan_bad_config_rejected():
    lib = _lib.lib()
    h = C.c_void_p()
    cfg = _hifigan_cfg()
    cfg.upsample_kernel_sizes[0] = 11  # (k=11,u=5) does not give u*L samples
    assert lib.mb_gan_create(C.byref(cfg), C.byref(h)) == 1
    assert b"upsample" in lib.mb_last_error()
    cfg = _hifigan_cfg()
    cfg.resblock_kernel_sizes[0] = 13
    assert lib.mb_gan_create(C.byref(cfg), C.byref(h)) == 1


def test_fregan_plan():
    from mockingbird_b200.vocoder.fregan.models import DEFAULT_CONFIG, FreGAN

    g = FreGAN(DEFAULT_CONFIG, precision="fp32")
    assert g.hop == 200
    infos = [g.layer_info(i) for i in range(g.num_layers())]
    assert sum("cond_up" in s for s in infos) == 4
    assert sum("res_output" in s for s in infos) == 3
    assert sum("resblocks" in s for s in infos) == 120  # SURVEY.md appendix A.2


def test_generator_without_cuda_fails_loudly():
    import torch
    from mockingbird_b200.vocoder.hifigan.models import DEFAULT_CONFIG_16K, Generator

    if torch.cuda.is_available():
        pytest.skip("CUDA present")
    g = Generator(DEFAULT_CONFIG_16K, precision="fp32")
    with pytest.raises(_lib.MbError):
        g.cuda()
    with pytest.raises(_lib.MbError):
        g.to("cpu")


def test_text_front_end_matches_reference_ids(golden_dir):
    """symbols table (utils/symbols.py:18) and basic_cleaners text_to_sequence (utils/text.py:13-40); the reference's ids
    are stored by oracle/make_golden_pinned.py"""
    from mockingbird_b200.synthesizer.utils.symbols import symbols
    from mockingbird_b200.synthesizer.utils.text import text_to_sequence

    assert len(symbols) == 75 and symbols[0] == "_" and symbols[1] == "~"
    assert text_to_sequence("Hello  World 1", ["basic_cleaners"]) == [35, 32, 39, 39, 42, 74, 50, 42, 45, 39, 31, 74, 54, 1]
    pinned = json.loads((golden_dir / "reference_pinned.json").read_text())
    for case in pinned["text_to_sequence"]:
        assert text_to_sequence(case["text"], ["basic_cleaners"]) == case["ids"], case["text"]


def test_tacotron_handle_and_missing_weight_errors():
    from mockingbird_b200.synthesizer.models.tacotron import Tacotron

    t = Tacotron(512, 75, 256, 128, 80, 80, 512, 5, 1024, 5, 4, 0.5, -3.4, 256)
    assert _lib.lib().mb_tacotron_arena_bytes(t._handle) > 32_000_000 * 4
    assert _lib.lib().mb_tacotron_workspace_bytes(t._handle, 2, 10, 20, 2) > 0
    assert _lib.lib().mb_tacotron_finalize(t._handle, None) == 2  # weights never set


def test_gan_plan_structure_on_cpu():
    """mb_gan_create is host-only: the lowering of the two generators can be checked without a GPU.
    HiFi-GAN: conv_pre + 4 x (ups + 3 resblocks x 3 x 2 convs) + conv_post = 78 ops.
    Fre-GAN (tensor-core path): the 16-channel full-rate stage is carried with 32 channels, `x += cond_up(mel)` is a
    separate add op for cond_up.1-3 (cond_up.0 reads the caller's fp32 mel and keeps the fused form); the FP32 path
    keeps the checkpoint's channel counts and the fused form everywhere."""
    import sys
    from pathlib import Path

    sys.path.insert(0, str(Path(__file__).resolve().parent.parent / "oracle"))
    import ref_init as ri
    from mockingbird_b200.vocoder.fregan.models import FreGAN
    from mockingbird_b200.vocoder.hifigan.models import Generator

    h = Generator(ri.HIFIGAN_CONFIG_16K, precision="f16tc")
    assert h.num_layers() == 78 and h.hop == 200
    tc = FreGAN(ri.FREGAN_CONFIG, precision="f16tc")
    info = [tc.layer_info(i) for i in range(tc.num_layers())]
    assert tc.hop == 200
    assert sum(s.startswith("add x+=cond_up.") for s in info) == 3 and not any("x+=cond_up.0" in s for s in info)
    assert any(s.startswith("conv resblocks.12.convs1.0 cin=32 cout=32") for s in info)
    assert any(s.startswith("conv conv_post cin=32 cout=1") for s in info)
    # the add follows its cond_up immediately and precedes the res_output / ups of the same stage
    i = next(k for k, s in enumerate(info) if s.startswith("conv cond_up.2"))
    assert info[i + 1].startswith("add x+=cond_up.2") and info[i + 2].startswith("conv res_output.1.1")
    f32 = FreGAN(ri.FREGAN_CONFIG, precision="fp32")
    info32 = [f32.layer_info(i) for i in range(f32.num_layers())]
    assert not any(s.startswith("add x+=") for s in info32)
    assert any(s.startswith("conv resblocks.12.convs1.0 cin=16 cout=16") for s in info32)
    assert len(info32) == len(info) - 3


def test_drop_in_surface_names_present():
    """INTEGRATION.md's import switch: every attribute the reference's callers use on these modules / classes exists
    (gen_voice.py:41, control/toolbox/__init__.py:215,283-344, control/mkgui/app.py:125)"""
    import numpy as np

    from mockingbird_b200.encoder import inference as enc
    from mockingbird_b200.synthesizer.inference import Synthesizer
    from mockingbird_b200.vocoder.fregan import inference as fre
    from mockingbird_b200.vocoder.hifigan import inference as gan
    from mockingbird_b200.vocoder.wavernn import inference as rnn

    for name in ("load_model", "is_loaded", "embed_utterance", "embed_frames_batch", "compute_partial_slices", "preprocess_wav"):
        assert callable(getattr(enc, name)), name
    for name in ("synthesize_spectrograms", "load_preprocess_wav", "make_spectrogram", "griffin_lim", "is_loaded", "load"):
        assert callable(getattr(Synthesizer, name)), name
    assert Synthesizer.sample_rate == 16000 and hasattr(Synthesizer, "hparams")
    for mod in (gan, fre, rnn):
        for name in ("load_model", "is_loaded", "infer_waveform"):
            assert callable(getattr(mod, name)), (mod.__name__, name)
    # host utilities run without a GPU
    wav = (np.sin(np.arange(16000) * 0.05) * 0.01).astype(np.float32)
    out = enc.preprocess_wav(wav, source_sr=16000, trim_silence=False)
    assert abs(10 * np.log10(np.mean(out ** 2)) - (-30)) < 1e-3       # normalised up to -30 dBFS
    assert enc.preprocess_wav(wav, source_sr=32000, normalize=False, trim_silence=False).shape[0] == 8000
    mel = np.random.RandomState(0).rand(80, 20).astype(np.float32) * 8 - 4
    y = Synthesizer.griffin_lim(mel)
    assert y.ndim == 1 and abs(len(y) - 19 * 256) <= 256 and np.isfinite(y).all()
