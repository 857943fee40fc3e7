"""The C-ABI library loads on a CPU-only box and exports every symbol include/funcodec_b200.h declares
(no compute calls without a GPU); host-side config logic matches the reference formulas."""
import ctypes
import os
import re

import pytest

from funcodec_b200 import _capi, get_config

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, "include", "funcodec_b200.h")).read()
    declared = set(re.findall(r"FCB_API\s+[\w\s\*]+?\b(fcb_\w+)\s*\(", hdr))
    assert declared, "no declarations parsed"
    assert declared == set(_capi.SYMBOLS), (declared ^ set(_capi.SYMBOLS))
    lib = _capi.load_library()
    for name in declared:
        assert hasattr(lib, name)
    assert lib.fcb_version().startswith(b"funcodec_b200")


def test_create_without_gpu_fails_loudly_not_silently():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from funcodec_b200.encodec import B200Encodec
    from funcodec_b200 import init_state_dict
    cfg = get_config("tiny_ds40")
    with pytest.raises(Exception):
        B200Encodec(cfg, init_state_dict(cfg, 0), "cuda:0")
    with pytest.raises(_capi.FcbError):
        B200Encodec(cfg, init_state_dict(cfg, 0), "cpu")


def test_bandwidth_to_quantizers():
    """vq.py:105-117 and codec_inference.py:121-125."""
    cfg = get_config("encodec_16k_n32_ds640")
    assert cfg.bandwidth_per_quantizer() == 250.0
    assert [cfg.num_quantizers_for_bandwidth(b) for b in (None, 0, 250, 499, 4000, 8000, 99999)] == [32, 32, 1, 1, 16, 32, 399]
    cfg = get_config("encodec_16k_n32_ds320")
    assert cfg.bandwidth_per_quantizer() == 500.0 and cfg.hop_length == 320 and cfg.frames(480000) == 1500


def test_config_from_reference_like_model():
    """integration.config_from_reference_model on a duck-typed stand-in for the reference Encodec module."""
    import types
    import torch
    from funcodec_b200 import init_state_dict
    from funcodec_b200.integration import config_from_reference_model, UnsupportedReferenceModel
    cfg = get_config("encodec_16k_n32_ds320")
    sd = init_state_dict(cfg, 0)
    m = types.SimpleNamespace(
        encoder=types.SimpleNamespace(ratios=list(reversed(cfg.ratios))), decoder=types.SimpleNamespace(ratios=list(cfg.ratios)),
        quantizer=types.SimpleNamespace(sampling_rate=16000, encoder_hop_length=320, codebook_size=1024, input_proj=None, input_act=None),
        audio_normalize=True, segment_dur=None, codec_domain="time", state_dict=lambda: sd)
    got = config_from_reference_model(m)
    for f in ("ratios", "n_filters", "dimension", "kernel_size", "last_kernel_size", "residual_kernel_size", "lstm_layers",
              "codebook_size", "num_quantizers", "sample_rate", "audio_normalize"):
        assert getattr(got, f) == getattr(cfg, f), f
    m.segment_dur = 1.0                     # segmenting is handled by the wrapper (fcb_roundtrip_segmented), not the config
    assert config_from_reference_model(m).ratios == cfg.ratios
    m.quantizer.input_proj = object()
    with pytest.raises(UnsupportedReferenceModel):
        config_from_reference_model(m)


def test_config_from_reference_like_freqcodec():
    """Same, for a mag_phase FreqCodec (codec_freq.py:118-215): [freq, time] ratio pairs, domain_conf."""
    import types
    from funcodec_b200 import init_state_dict
    from funcodec_b200.integration import config_from_reference_model, UnsupportedReferenceModel
    cfg = get_config("freq_small")
    sd = init_state_dict(cfg, 0)
    pairs = [[f, t] for f, t in zip(cfg.ratios_f, cfg.ratios)]
    m = types.SimpleNamespace(
        encoder=types.SimpleNamespace(ratios=list(reversed(pairs))), decoder=types.SimpleNamespace(ratios=pairs),
        quantizer=types.SimpleNamespace(sampling_rate=cfg.sample_rate, encoder_hop_length=cfg.hop_length,
                                        codebook_size=cfg.codebook_size, input_proj=None, input_act=None),
        audio_normalize=True, segment_dur=None, codec_domain=["mag_phase", "mag_phase"],
        domain_conf={"n_fft": cfg.n_fft, "hop_length": cfg.stft_hop}, state_dict=lambda: sd)
    got = config_from_reference_model(m)
    for f in ("arch", "ratios", "ratios_f", "n_fft", "stft_hop", "n_filters", "dimension", "kernel_size", "last_kernel_size",
              "residual_kernel_size", "lstm_layers", "codebook_size", "num_quantizers"):
        assert getattr(got, f) == getattr(cfg, f), f
    assert (got.conv_group_ratio, got.tr_conv_group_ratio) == (-1, -1)
    # grouped 2-D convs: the ratios are recovered from the weight shapes
    gcfg = get_config("freq_small_grouped")
    gsd = init_state_dict(gcfg, 0)
    m.state_dict = lambda: gsd
    got = config_from_reference_model(m)
    assert (got.conv_group_ratio, got.tr_conv_group_ratio, got.n_filters) == (gcfg.conv_group_ratio, gcfg.tr_conv_group_ratio, gcfg.n_filters)
    m.state_dict = lambda: sd
    m.segment_dur = 1.0
    with pytest.raises(UnsupportedReferenceModel):
        config_from_reference_model(m)
    m.segment_dur = None
    m.codec_domain = ["stft", "stft"]
    with pytest.raises(UnsupportedReferenceModel):
        config_from_reference_model(m)


def reference_description():
    """tests/golden/reference_modules.json.gz: the reference's own module trees, attributes and state_dict shapes
    (tools/gen_golden_reference_modules.py)."""
    import gzip
    import json
    with gzip.open(os.path.join(ROOT, "tests", "golden", "reference_modules.json.gz"), "rt") as f:
        return json.load(f)


def rebuild_reference_encodec(desc):
    """A stand-in for the reference `Encodec` rebuilt from its recorded description: encoder / decoder module trees with the
    recorded class names and attributes (torch's own GroupNorm / ELU / Sequential where the reference uses them), the
    quantizer attributes, and a state_dict of meta tensors with the recorded names and shapes."""
    import types
    import torch
    import torch.nn as nn
    classes = {}

    def make(cls, attrs):
        if cls == "GroupNorm":
            return nn.GroupNorm(attrs["num_groups"], attrs["num_channels"], attrs["eps"], attrs["affine"])
        if cls == "ELU":
            return nn.ELU(attrs["alpha"])
        mod = nn.Sequential() if cls == "Sequential" else classes.setdefault(cls, type(cls, (nn.Module,), {}))()
        for k, v in attrs.items():
            setattr(mod, k, v)
        return mod

    def tree(entries):
        root = make(entries[0][1], entries[0][2])
        for path, cls, attrs in entries[1:]:
            parent, _, leaf = path.rpartition(".")
            root.get_submodule(parent).add_module(leaf, make(cls, attrs))
        return root

    sd = {k: torch.empty(shape, device="meta") for k, shape in desc["state_dict"].items()}
    return types.SimpleNamespace(
        encoder=tree(desc["encoder"]), decoder=tree(desc["decoder"]),
        quantizer=types.SimpleNamespace(rq=types.SimpleNamespace(model=types.SimpleNamespace(**desc["rq_model"])),
                                        **desc["quantizer"]),
        state_dict=lambda: sd, **desc["attrs"])


def test_config_from_the_real_reference_modules():
    """integration.config_from_reference_model + state_dict name coverage on the REAL reference `Encodec` (as recorded in
    tests/golden/reference_modules.json.gz from the models tools/ref_harness.py builds): every field matches the preset, every
    tensor the engine needs is in the reference's state_dict under the same name and shape, and option variants that keep
    the shapes are refused."""
    from funcodec_b200.integration import config_from_reference_model, stacked_codebooks, UnsupportedReferenceModel
    from funcodec_b200.weights import state_dict_shapes
    models = reference_description()["models"]
    for name in ("encodec_16k_n32_ds320", "tiny_ds40", "soundstream_noncausal_small", "soundstream_causal_small",
                 "weightnorm_lstm_small"):
        cfg = get_config(name)
        m = rebuild_reference_encodec(models[name])
        got = config_from_reference_model(m)
        for f in ("arch", "ratios", "n_filters", "dimension", "kernel_size", "last_kernel_size", "residual_kernel_size",
                  "lstm_layers", "codebook_size", "num_quantizers", "sample_rate", "audio_normalize", "n_residual_layers",
                  "dilation_base", "norm", "causal"):
            assert getattr(got, f) == getattr(cfg, f), (name, f)
        sd = m.state_dict()
        for k, shp in state_dict_shapes(cfg).items():
            assert k in sd and tuple(sd[k].shape) == tuple(shp), (name, k)
        assert tuple(stacked_codebooks(sd).shape) == (cfg.num_quantizers, cfg.codebook_size, cfg.dimension)
    # options that keep parameter names and shapes but change the maths are refused
    m = rebuild_reference_encodec(models["tiny_ds40"])
    m.encoder.model[0].causal = True                   # one causal conv among non-causal ones / causal under GroupNorm
    with pytest.raises(UnsupportedReferenceModel):
        config_from_reference_model(m)
    m.encoder.model[0].causal = False
    m.decoder.model[0].pad_mode = "constant"
    with pytest.raises(UnsupportedReferenceModel):
        config_from_reference_model(m)
    m.decoder.model[0].pad_mode = "reflect"
    m.quantizer.rq.model.q0_ds_ratio = 2
    with pytest.raises(UnsupportedReferenceModel):
        config_from_reference_model(m)


def test_use_ddp_false_reference_quantizer_keys():
    """`use_ddp: false` (core_vq.py:147-150): the reference's own per-layer key names are what stacked_codebooks / fcb_finalize
    assemble into the [n_q, K, D] codebook tensor."""
    import torch
    from funcodec_b200.integration import stacked_codebooks
    # (in the reference CostumeQuantizer(use_ddp=False) itself raises -- vq.py:73-84 passes q0_ds_ratio, which
    # core_vq.VectorQuantization does not accept -- so the fixture records the RVQ class built directly
    # (3 layers, dim 16, 32 codes); it sits at quantizer.rq.model)
    keys = reference_description()["rvq_use_ddp_false"]
    sd = {"quantizer.rq.model." + k: torch.zeros(shape) for k, shape in keys.items()}
    assert "quantizer.rq.model.layers.0._codebook.embed" in sd and "quantizer.rq.model.embed" not in sd
    for i in range(3):
        sd[f"quantizer.rq.model.layers.{i}._codebook.embed"] = torch.full((32, 16), float(i))
    e = stacked_codebooks(sd)
    assert tuple(e.shape) == (3, 32, 16) and [float(e[i, 0, 0]) for i in range(3)] == [0.0, 1.0, 2.0]
