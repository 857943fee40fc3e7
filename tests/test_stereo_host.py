"""Stereo (two-channel) time-domain Encodec, host side (CPU): the preset, the YAML and reference-module mappings, the CLI's
refusal of stereo file I/O, the weight shapes and the analytic work model."""
import dataclasses
import os
import types

import pytest
import yaml

from funcodec_b200 import get_config, init_state_dict, state_dict_shapes
from funcodec_b200.bin import codec_inference as CLI
from funcodec_b200.integration import UnsupportedReferenceModel, config_from_reference_model
from funcodec_b200.workload import conv_launches, workload_model

FIELDS = ("arch", "ratios", "n_filters", "dimension", "kernel_size", "last_kernel_size", "residual_kernel_size", "lstm_layers",
          "codebook_size", "num_quantizers", "sample_rate", "audio_normalize", "hop_length", "n_residual_layers",
          "dilation_base", "norm", "causal", "channels")


def _stereo_yaml(cfg, tmp_path, input_size=2, dec_channels=2):
    conf = dict(norm=cfg.norm, causal=cfg.causal, ratios=list(cfg.ratios), n_filters=cfg.n_filters,
                seq_layer_num=cfg.lstm_layers, n_residual_layers=cfg.n_residual_layers, dilation_base=cfg.dilation_base)
    if cfg.lstm_layers == 0:
        conf["seq_model"] = "none"
    a = dict(input_size=input_size, model="encodec", encoder_conf=dict(conf), decoder_conf=dict(conf, channels=dec_channels),
             quantizer_conf=dict(codebook_size=cfg.codebook_size, num_quantizers=cfg.num_quantizers, sampling_rate=cfg.sample_rate,
                                 encoder_hop_length=cfg.hop_length, use_ddp=True),
             model_conf=dict(odim=cfg.dimension, audio_normalize=True, segment_dur=None, overlap_ratio=None))
    path = os.path.join(str(tmp_path), "config.yaml")
    with open(path, "wt") as f:
        yaml.safe_dump(a, f)
    return path


def test_stereo_preset_is_the_48k_layout():
    cfg = get_config("encodec_48k_stereo")
    assert (cfg.sample_rate, cfg.ratios, cfg.n_filters, cfg.dimension, cfg.lstm_layers, cfg.codebook_size, cfg.num_quantizers,
            cfg.norm, cfg.causal, cfg.channels) == (48000, (8, 5, 4, 2), 32, 128, 2, 1024, 16, "time_group_norm", False, 2)
    assert cfg.hop_length == 320 and cfg.frames(48000) == 150


@pytest.mark.parametrize("name", ["encodec_48k_stereo", "stereo_small", "stereo_causal_small"])
def test_config_from_yaml_roundtrips_the_stereo_presets(tmp_path, name):
    cfg = get_config(name)
    got, seg, ov = CLI.config_from_yaml(_stereo_yaml(cfg, tmp_path))
    for f in FIELDS:
        assert getattr(got, f) == getattr(cfg, f), f
    assert seg is None and ov is None


@pytest.mark.parametrize("input_size, dec_channels", [(2, 1), (1, 2), (3, 3)])
def test_config_from_yaml_refuses_unbuilt_channel_layouts(tmp_path, input_size, dec_channels):
    with pytest.raises(SystemExit, match="unsupported configuration"):
        CLI.config_from_yaml(_stereo_yaml(get_config("stereo_small"), tmp_path, input_size, dec_channels))


def test_cli_refuses_a_stereo_yaml(tmp_path):
    """wav.scp / PCM16 I/O is mono: a stereo model through the CLI stops with a message naming B200Encodec, before any model
    file is read or a GPU is touched."""
    path = _stereo_yaml(get_config("encodec_48k_stereo"), tmp_path)
    argv = ["--data_path_and_name_and_type", f"{tmp_path}/wav.scp,speech,sound", "--config_file", path,
            "--model_file", f"{tmp_path}/missing.pth", "--output_dir", f"{tmp_path}/out", "--sampling_rate", "48000"]
    with pytest.raises(SystemExit, match="unsupported configuration.*B200Encodec"):
        CLI.main(argv)
    with pytest.raises(SystemExit, match="unsupported configuration"):
        CLI.build_speech2token(path, f"{tmp_path}/missing.pth")


def test_stereo_weight_shapes():
    for name in ("encodec_48k_stereo", "stereo_causal_small"):
        cfg = get_config(name)
        sh = state_dict_shapes(cfg)
        wk = "weight_v" if cfg.norm == "weight_norm" else "weight"
        last = max(int(k.split(".")[2]) for k in sh if k.startswith("decoder.model."))
        assert sh["encoder.model.0.conv.conv." + wk] == (cfg.n_filters, 2, cfg.kernel_size)
        assert sh[f"decoder.model.{last}.conv.conv.{wk}"] == (2, cfg.n_filters, cfg.last_kernel_size)
        assert sh[f"decoder.model.{last}.conv.conv.bias"] == (2,)
        if cfg.norm == "time_group_norm":
            assert sh[f"decoder.model.{last}.conv.norm.weight"] == sh[f"decoder.model.{last}.conv.norm.bias"] == (2,)
        mono = state_dict_shapes(dataclasses.replace(cfg, channels=1))
        diff = {k for k in sh if sh[k] != mono[k]}
        assert diff <= {"encoder.model.0.conv.conv." + wk, f"decoder.model.{last}.conv.conv.{wk}",
                        f"decoder.model.{last}.conv.conv.bias", f"decoder.model.{last}.conv.norm.weight",
                        f"decoder.model.{last}.conv.norm.bias", f"decoder.model.{last}.conv.conv.weight_g"}


def _reference_like(cfg, enc_channels, dec_channels):
    """A stand-in with the attributes config_from_reference_model reads off SEANetEncoder / SEANetDecoder / CostumeQuantizer /
    Encodec (plain objects: no module options to inspect)."""
    sd = init_state_dict(cfg, 0)
    return types.SimpleNamespace(
        encoder=types.SimpleNamespace(ratios=list(reversed(cfg.ratios)), channels=enc_channels),
        decoder=types.SimpleNamespace(ratios=list(cfg.ratios), channels=dec_channels),
        quantizer=types.SimpleNamespace(sampling_rate=cfg.sample_rate, encoder_hop_length=cfg.hop_length),
        audio_normalize=cfg.audio_normalize, codec_domain="time", state_dict=lambda: sd)


def test_config_from_reference_model_reads_the_channels():
    for name in ("encodec_48k_stereo", "stereo_small"):
        cfg = get_config(name)
        got = config_from_reference_model(_reference_like(cfg, 2, 2))
        for f in FIELDS:
            assert getattr(got, f) == getattr(cfg, f), (name, f)
    mono = get_config("tiny_ds40")
    assert config_from_reference_model(_reference_like(mono, 1, 1)).channels == 1
    with pytest.raises(UnsupportedReferenceModel, match="channels"):
        config_from_reference_model(_reference_like(get_config("stereo_small"), 2, 1))


def test_workload_mono_unchanged_and_stereo_layers_by_hand():
    for name in ("encodec_16k_n32_ds640", "encodec_16k_n32_ds320", "soundstream_16k_n32_ds320", "tiny_ds40"):
        cfg = get_config(name)
        assert workload_model(cfg, 16000) == workload_model(dataclasses.replace(cfg, channels=1), 16000)
    cfg = get_config("encodec_48k_stereo")
    mono = dataclasses.replace(cfg, channels=1)
    L = 48000
    st, mo = conv_launches(cfg, L), conv_launches(mono, L)
    assert [l["name"] for l in st] == [l["name"] for l in mo]
    nf, k = cfg.n_filters, cfg.kernel_size
    # first conv: 2 -> 32 channels, k 7, stride 1 over L samples (padded input L + 6)
    first = st[0]
    assert first["name"] == "enc.conv0" and (first["cin"], first["cout"]) == (2, nf)
    assert first["macs"] == L * 2 * nf * k and first["bytes"] == 4 * ((L + k - 1) * 2 + L * nf)
    # last conv: 32 -> 2 channels, k 7 over the decoded T' * hop samples
    last = st[-1]
    T = cfg.frames(L) * cfg.hop_length
    kl = cfg.last_kernel_size
    assert last["name"] == "dec.final" and (last["cin"], last["cout"]) == (nf, 2)
    assert last["macs"] == T * nf * 2 * kl and last["bytes"] == 4 * ((T + kl - 1) * nf + T * 2)
    assert all(a == b for a, b in zip(st[1:-1], mo[1:-1]))
    ws, wm = workload_model(cfg, L), workload_model(mono, L)
    assert ws["conv_macs"] - wm["conv_macs"] == L * nf * k + T * nf * kl
    assert ws["conv_bytes"] - wm["conv_bytes"] == 4 * ((L + k - 1) + T)
    assert ws["conv_params"] - wm["conv_params"] == nf * k + nf * kl + 1 + 2
