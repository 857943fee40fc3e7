"""The `encoding_decoding.sh` drop-in CLI (funcodec_b200/bin/codec_inference.py) and its host plumbing.

CPU: the literal argument lists of the script's three stages parse; the reference's YAMLs map to the presets; key_file
sharding, codecs.txt / Kaldi ark outputs and the three run modes work end to end with the ORACLE behind the Speech2Token call
signature (test infrastructure only).  GPU: the same command lines through main() on the CUDA library."""
import json
import os

import numpy as np
import pytest
import torch

from funcodec_b200 import get_config, init_state_dict, pipeline as P
from funcodec_b200.bin import codec_inference as CLI
from funcodec_b200.kaldi_io import ArkScpWriter, read_mat, read_scp_mats

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def stage_argv(stage, d, job=1, batch_size=4, bit_width=16000, indices_save_type="text", sr=16000):
    """egs/LibriTTS/codec/encoding_decoding.sh:80-98 (stage 1), :124-143 (stage 2), :168-187 (stage 3), verbatim flag order."""
    src, fmt, mod, need = {1: ("wav.scp", "sound", "encode", "true"), 2: ("codecs.txt", "codec_json", "decode", "false"),
                           3: ("emb.scp", "kaldi_ark", "decode_emb", "false")}[stage]
    a = ["--batch_size", str(batch_size), "--num_workers", "4", "--ngpu", "1", "--gpuid_list", "0",
         "--data_path_and_name_and_type", f"{d}/{src},speech,{fmt}", "--key_file", f"{d}/logdir/keys.{job}.scp",
         "--config_file", f"{d}/model/config.yaml", "--model_file", f"{d}/model/model.pth",
         "--output_dir", f"{d}/logdir/output.{job}", "--sampling_rate", str(sr), "--file_sampling_rate", str(sr),
         "--bit_width", str(bit_width), "--need_indices", need, "--need_sub_quants", "false", "--use_scale", "false"]
    if stage == 1:
        a += ["--indices_save_type", indices_save_type]
    return a + ["--run_mod", mod]


def test_parser_accepts_the_scripts_literal_argv_and_has_the_reference_defaults():
    p = CLI.get_parser()
    for stage in (1, 2, 3):
        a = p.parse_args(stage_argv(stage, "/x"))
        assert a.run_mod == {1: "encode", 2: "decode", 3: "decode_emb"}[stage]
        assert a.key_file == "/x/logdir/keys.1.scp" and a.use_scale is False and a.need_sub_quants is False
        assert a.data_path_and_name_and_type[0][2] == {1: "sound", 2: "codec_json", 3: "kaldi_ark"}[stage]
    d = p.parse_args([])
    # codec_inference.py:428-558
    assert (d.use_scale, d.bit_width, d.batch_size, d.sampling_rate, d.indices_save_type, d.run_mod, d.dtype, d.ngpu) == \
        (True, 16000, 1, 24000, "text", "inference", "float32", 0)
    assert d.need_indices is None and d.key_file is None
    # job id = suffix of --output_dir picks the GPU round-robin (codec_inference.py:565-575)
    assert [CLI.pick_gpu(f"/x/output.{j}", "4,5,6") for j in (1, 2, 3, 4)] == [4, 5, 6, 4]
    assert CLI.pick_gpu(None, "") == 0


def _yaml_for(cfg, tmp_path, **model_conf):
    import yaml
    if cfg.arch == 1:
        ratios = [[f, t] for f, t in zip(cfg.ratios_f, cfg.ratios)]
        model, extra = "freq_codec", dict(codec_domain=["mag_phase", "mag_phase"])
    else:
        ratios, model, extra = list(cfg.ratios), "encodec", {}
    conf = dict(norm=cfg.norm, causal=cfg.causal, ratios=ratios, n_filters=cfg.n_filters,
                seq_layer_num=cfg.lstm_layers, n_residual_layers=cfg.n_residual_layers, dilation_base=cfg.dilation_base)
    if cfg.norm == "time_group_norm":
        conf["norm_params"] = dict(num_groups=1)
    if cfg.lstm_layers == 0:
        conf["seq_model"] = "none"
    if cfg.conv_group_ratio > 0:
        conf["conv_group_ratio"] = cfg.conv_group_ratio
    a = dict(encoder_conf=dict(conf), decoder_conf=dict(conf), model=model,
             quantizer_conf=dict(codebook_size=cfg.codebook_size, num_quantizers=cfg.num_quantizers, sampling_rate=cfg.sample_rate,
                                 encoder_hop_length=cfg.hop_length, use_ddp=True),
             model_conf=dict(odim=cfg.dimension, audio_normalize=True, segment_dur=None, overlap_ratio=None, **extra, **model_conf))
    if cfg.tr_conv_group_ratio > 0:
        a["decoder_conf"]["tr_conv_group_ratio"] = cfg.tr_conv_group_ratio
    path = os.path.join(tmp_path, "config.yaml")
    with open(path, "wt") as f:
        yaml.safe_dump(a, f)
    return path


@pytest.mark.parametrize("name", ["encodec_16k_n32_ds640", "encodec_16k_n32_ds320", "tiny_ds40", "freqcodec_magphase_16k_n32_ds320",
                                  "freqcodec_magphase_16k_n32_ds320_gr8", "freq_small_grouped", "soundstream_noncausal_16k_n32_ds640",
                                  "soundstream_16k_n32_ds320", "soundstream_causal_small", "weightnorm_lstm_small"])
def test_config_from_yaml_roundtrips_the_presets(tmp_path, name):
    cfg = get_config(name)
    got, seg, ov = CLI.config_from_yaml(_yaml_for(cfg, str(tmp_path)))
    for f in ("arch", "ratios", "ratios_f", "n_filters", "dimension", "kernel_size", "last_kernel_size", "residual_kernel_size",
              "lstm_layers", "codebook_size", "num_quantizers", "sample_rate", "audio_normalize", "conv_group_ratio",
              "tr_conv_group_ratio", "n_fft", "stft_hop", "hop_length", "n_residual_layers", "dilation_base", "norm", "causal"):
        assert getattr(got, f) == getattr(cfg, f), f
    assert seg is None and ov is None


@pytest.mark.parametrize("patch", [dict(norm="layer_norm"), dict(norm="spectral_norm"), dict(norm="time_group_norm", causal=True),
                                   dict(trim_right_ratio=0.5), dict(pad_mode="constant"), dict(activation="ReLU")])
def test_config_from_yaml_refuses_unbuilt_conv_options(tmp_path, patch):
    """norm outside {time_group_norm, weight_norm, none}, causal under GroupNorm (the reference itself raises, conv.py:46-47),
    partial right trimming, other paddings / activations: refused with a message, never approximated."""
    import yaml
    path = _yaml_for(get_config("weightnorm_lstm_small"), str(tmp_path))
    with open(path) as f:
        a = yaml.safe_load(f)
    for side in ("encoder_conf", "decoder_conf"):
        a[side].update(patch)
    with open(path, "wt") as f:
        yaml.safe_dump(a, f)
    with pytest.raises(SystemExit, match="unsupported configuration"):
        CLI.config_from_yaml(path)


def test_config_from_the_reference_repo_yamls(tmp_path):
    """The YAMLs the reference ships (egs/LibriTTS/codec/conf, as recorded in tests/golden/reference_modules.json.gz): the two
    Encodec ones, the two mag_phase FreqCodec ones, the two non-causal SoundStream ones (3 dilated residual blocks per stage,
    no sequence model) and the causal weight_norm SoundStream one map to presets; the mag_angle FreqCodec one is refused with
    a message."""
    import gzip
    import yaml
    with gzip.open(os.path.join(ROOT, "tests", "golden", "reference_modules.json.gz"), "rt") as f:
        confs = json.load(f)["yaml_conf"]
    assert len(confs) == 8
    want = {"encodec_16k_n32_600k_step.yaml": "encodec_16k_n32_ds320", "encodec_16k_n32_600k_step_ds640.yaml": "encodec_16k_n32_ds640",
            "soundstream_noncausal_16k_n32_600k_step.yaml": "soundstream_noncausal_16k_n32_ds320",
            "soundstream_noncausal_16k_n32_600k_step_ds640.yaml": "soundstream_noncausal_16k_n32_ds640",
            "soundstream_16k_n32_600k_step.yaml": "soundstream_16k_n32_ds320",
            "freqcodec_mag_phase_16k_n32_600k_step.yaml": "freqcodec_magphase_16k_n32_ds320",
            "freqcodec_mag_phase_16k_n32_600k_step_ds640.yaml": "freqcodec_magphase_16k_n32_ds640"}
    for fn in sorted(confs):
        path = os.path.join(tmp_path, fn)
        with open(path, "wt") as f:
            yaml.safe_dump(confs[fn], f)
        if fn in want:
            got, _, _ = CLI.config_from_yaml(path)
            cfg = get_config(want[fn])
            for f in ("arch", "ratios", "ratios_f", "n_filters", "dimension", "lstm_layers", "codebook_size", "num_quantizers",
                      "sample_rate", "hop_length", "conv_group_ratio", "n_residual_layers", "dilation_base", "norm", "causal"):
                assert getattr(got, f) == getattr(cfg, f), (fn, f)
        else:
            with pytest.raises(SystemExit):
                CLI.config_from_yaml(path)


def test_kaldi_ark_scp_format(tmp_path):
    """Byte layout of kaldiio's float-matrix ark + scp offsets (what the reference's WriteHelper("ark,scp,f:...") emits)."""
    pre = os.path.join(tmp_path, "m")
    a = np.arange(6, dtype=np.float32).reshape(2, 3)
    b = np.linspace(-1, 1, 8, dtype=np.float32).reshape(4, 2)
    with ArkScpWriter(pre) as w:
        w("utt_a", a)
        w("utt_b", b)
    raw = open(pre + ".ark", "rb").read()
    assert raw.startswith(b"utt_a \0BFM \x04\x02\x00\x00\x00\x04\x03\x00\x00\x00" + a.tobytes() + b"utt_b \0BFM ")
    lines = open(pre + ".scp").read().split("\n")
    assert lines[0] == f"utt_a {pre}.ark:6" and lines[1] == f"utt_b {pre}.ark:{6 + 15 + 24 + 6}"
    got = dict(read_scp_mats(pre + ".scp"))
    assert np.array_equal(got["utt_a"], a) and np.array_equal(got["utt_b"], b)
    assert np.array_equal(read_mat(f"{pre}.ark:6"), a)


def _write_corpus(d, cfg, lens, seed=5):
    os.makedirs(os.path.join(d, "logdir"), exist_ok=True)
    g = torch.Generator().manual_seed(seed)
    clips = {}
    with open(os.path.join(d, "wav.scp"), "wt") as f:
        for i, n in enumerate(lens):
            x = (0.3 * torch.randn(n, generator=g)).clamp(-0.99, 0.99)
            path = os.path.join(d, f"u{i}.wav")
            P.save_wav_pcm16(path, x.view(1, -1), cfg.sample_rate, rescale=False)
            clips[f"u{i}"] = P.load_wav(path)[0]
            f.write(f"u{i} {path}\n")
    # utils/split_scp.pl: contiguous shards of the key file
    keys = [f"u{i}" for i in range(len(lens))]
    half = (len(keys) + 1) // 2
    for job, ks in ((1, keys[:half]), (2, keys[half:])):
        with open(os.path.join(d, "logdir", f"keys.{job}.scp"), "wt") as f:
            for k in ks:
                f.write(f"{k} {os.path.join(d, k + '.wav')}\n")
    return clips


def test_three_stages_with_key_file_sharding_on_the_oracle(tmp_path):
    """Stage 1 (two JOB shards, text and ark index outputs) -> cat codecs.txt -> stage 2 -> stage 3 with the oracle behind
    Speech2Token's signature: exercises select_keys, IndicesWriter, sub-quants ark, run_decode, run_decode_emb."""
    from laura_calls import OracleSpeech2Token
    from oracle.encodec_oracle import OracleEncodec
    cfg = get_config("tiny_ds40")
    sd = init_state_dict(cfg, 3)
    ora = OracleEncodec(sd, cfg.ratios, cfg.sample_rate, cfg.lstm_layers)
    s2t = OracleSpeech2Token(ora)
    import types
    s2t.model = types.SimpleNamespace(quantizer=types.SimpleNamespace(encoder_hop_length=cfg.hop_length, sampling_rate=cfg.sample_rate))
    d = str(tmp_path)
    lens = [40 * 9 + 5, 40 * 14, 40 * 6 + 39, 40 * 11]
    clips = _write_corpus(d, cfg, lens)
    total = 0
    for job in (1, 2):
        out = os.path.join(d, "logdir", f"output.{job}")
        total += P.run_encode(s2t, os.path.join(d, "wav.scp"), out, batch_size=2, run_mod="encode", use_scale=False,
                              key_file=os.path.join(d, "logdir", f"keys.{job}.scp"), need_indices=True, need_sub_quants=True)
        assert not [f for f in os.listdir(out) if f.endswith(".wav")]           # encode mode writes no audio
    assert total == 4
    lines = []
    for job in (1, 2):
        lines += open(os.path.join(d, "logdir", f"output.{job}", "codecs.txt")).read().strip().split("\n")
    assert [l.split(" ", 1)[0] for l in lines] == ["u0", "u1", "u2", "u3"]
    with open(os.path.join(d, "codecs.txt"), "wt") as f:
        f.write("\n".join(lines) + "\n")
    # job 1's batch is (u0, u1) wrap-padded together: same codes as the oracle run directly
    speech, _ = P.wrap_pad_batch([clips["u0"], clips["u1"]])
    ref = ora.inference(speech, need_recon=False)["code_indices"][0]
    for i in range(2):
        key, arr = P.parse_indices_line(lines[i])
        tf = -(-lens[i] // cfg.hop_length)
        assert arr.shape == (tf, cfg.num_quantizers) and np.array_equal(arr, ref[:, i, :tf].numpy().T)
    sq = dict(read_scp_mats(os.path.join(d, "logdir", "output.1", "codec_emb.scp")))
    assert sq["u0"].shape == (-(-lens[0] // cfg.hop_length), cfg.num_quantizers * cfg.dimension)
    # ark indices: [T', n_q] float matrix with the same integers
    out_ark = os.path.join(d, "ark")
    P.run_encode(s2t, os.path.join(d, "wav.scp"), out_ark, batch_size=2, run_mod="encode", need_indices=True,
                 indices_save_type="ark", key_file=os.path.join(d, "logdir", "keys.1.scp"))
    m = dict(read_scp_mats(os.path.join(out_ark, "indices.scp")))
    assert np.array_equal(m["u1"], P.parse_indices_line(lines[1])[1].astype(np.float32))
    # need_indices false: nothing is written
    out_none = os.path.join(d, "none")
    P.run_encode(s2t, os.path.join(d, "wav.scp"), out_none, batch_size=4, run_mod="encode", need_indices=False)
    assert os.listdir(out_none) == []
    # stage 2 on shard 2 only
    dec = os.path.join(d, "dec")
    assert P.run_decode(s2t, os.path.join(d, "codecs.txt"), dec, batch_size=3, bit_width=16000,
                        key_file=os.path.join(d, "logdir", "keys.2.scp")) == 2
    assert sorted(os.listdir(dec)) == ["u2.wav", "u3.wav"]
    y, sr = P.load_wav(os.path.join(dec, "u2.wav"))
    assert sr == cfg.sample_rate and y.shape[0] == -(-lens[2] // cfg.hop_length) * cfg.hop_length
    # stage 3: embeddings [T', D] from a Kaldi scp
    with ArkScpWriter(os.path.join(d, "emb")) as w:
        for i, key in enumerate(["u0", "u1"]):
            e = ora.inference(torch.from_numpy(clips[key]).view(1, -1), need_recon=False)["code_embeddings"][0][0]
            w(key, e[0].numpy())
    dec3 = os.path.join(d, "dec3")
    assert P.run_decode_emb(s2t, os.path.join(d, "emb.scp"), dec3, batch_size=1) == 2
    y, _ = P.load_wav(os.path.join(dec3, "u1.wav"))
    assert y.shape[0] == 14 * cfg.hop_length
    with pytest.raises(KeyError):
        P.select_keys([("a", 1)], os.path.join(d, "logdir", "keys.1.scp"))


def test_main_refuses_before_touching_the_gpu():
    """Argument combinations this path does not serve end in SystemExit with a message before any model is built."""
    base = ["--data_path_and_name_and_type", "codecs.txt,codec,codec_json", "--output_dir", "/tmp/x/output.1",
            "--config_file", "/nonexistent.yaml", "--model_file", "/nonexistent.pth", "--sampling_rate", "16000"]
    with pytest.raises(SystemExit, match="inference / encode"):
        CLI.main(base + ["--file_sampling_rate", "8000", "--run_mod", "decode"])
    with pytest.raises(SystemExit, match="float32"):
        CLI.main(base + ["--dtype", "float16"])
    with pytest.raises(SystemExit, match="model_tag"):
        CLI.main(base + ["--model_tag", "damo/x"])


def test_inference_modelscope_callable_on_the_oracle(tmp_path):
    """`inference_modelscope(...)` -> `_forward(data | raw_inputs, output_dir_v2, param_dict)` (codec_inference.py:164-382) with the
    oracle behind Speech2Token's signature: the in-memory result list (no output directory), raw samples / a wav path as
    `raw_inputs`, files under `output_dir_v2`, the per-call `param_dict` bit_width, the three run_mods and `inference()`."""
    import types
    from laura_calls import OracleSpeech2Token
    from oracle.encodec_oracle import OracleEncodec
    cfg = get_config("tiny_ds40")
    sd = init_state_dict(cfg, 3)
    ora = OracleEncodec.from_config(sd, cfg)
    s2t = OracleSpeech2Token(ora)
    s2t.model = types.SimpleNamespace(quantizer=types.SimpleNamespace(encoder_hop_length=cfg.hop_length, sampling_rate=cfg.sample_rate))
    d = str(tmp_path)
    lens = [40 * 9 + 5, 40 * 14, 40 * 6 + 39]
    clips = _write_corpus(d, cfg, lens)
    bw_all = int(cfg.num_quantizers * cfg.bandwidth_per_quantizer())
    common = dict(batch_size=2, sampling_rate=cfg.sample_rate, bit_width=bw_all, use_scale=True, speech2token=s2t)
    fwd = CLI.inference_modelscope(output_dir=None, **common)
    # (a) data files, no output dir -> [{"key", "value"}] in file order, each trimmed to its own length
    res = fwd([(os.path.join(d, "wav.scp"), "speech", "sound")])
    assert [r["key"] for r in res] == ["u0", "u1", "u2"]
    assert [tuple(r["value"].shape) for r in res] == [(1, n) for n in lens]
    speech, _ = P.wrap_pad_batch([clips["u0"], clips["u1"]])
    ref = ora.inference(speech, need_recon=True, bit_width=bw_all, use_scale=True)["recon_speech"]
    assert torch.equal(res[1]["value"], ref[1][:, :lens[1]])
    # (b) raw samples and a wav path as raw_inputs
    one = fwd(raw_inputs=clips["u2"])
    ref2 = ora.inference(torch.from_numpy(clips["u2"]).view(1, -1), need_recon=True, bit_width=bw_all)["recon_speech"]
    assert len(one) == 1 and one[0]["key"] == "utt" and torch.equal(one[0]["value"], ref2[0])
    one = fwd(raw_inputs=torch.from_numpy(clips["u2"]))
    assert torch.equal(one[0]["value"], ref2[0])
    one = fwd(raw_inputs=os.path.join(d, "u2.wav"))
    assert one[0]["key"] == "u2" and torch.equal(one[0]["value"], ref2[0])
    # (c) param_dict: per-call bit width (fewer quantizers -> a different waveform), need_indices + output_dir_v2 -> files
    low = int(2 * cfg.bandwidth_per_quantizer())
    out = os.path.join(d, "out_v2")
    assert fwd([(os.path.join(d, "wav.scp"), "speech", "sound")], output_dir_v2=out,
               param_dict=dict(bit_width=low, need_indices=True)) == []
    assert sorted(os.listdir(out)) == ["codecs.txt", "u0.wav", "u1.wav", "u2.wav"]
    key, arr = P.parse_indices_line(open(os.path.join(out, "codecs.txt")).readline())
    assert key == "u0" and arr.shape == (-(-lens[0] // cfg.hop_length), 2)
    # (d) decode from the codes just written, decode_emb from embeddings, through fresh pipelines (run_mod is a pipeline kwarg)
    dec = CLI.inference_modelscope(output_dir=os.path.join(d, "dec"), run_mod="decode", **common)
    assert dec([(os.path.join(out, "codecs.txt"), "codec", "codec_json")]) == []
    y, sr = P.load_wav(os.path.join(d, "dec", "u1.wav"))
    assert sr == cfg.sample_rate and y.shape[0] == -(-lens[1] // cfg.hop_length) * cfg.hop_length
    mem = CLI.inference_modelscope(output_dir=None, run_mod="decode", **common)
    r = mem(raw_inputs=arr)                                   # codes [T', n_q] as raw input
    assert tuple(r[0]["value"].shape) == (1, arr.shape[0] * cfg.hop_length)
    with pytest.raises(ValueError):
        dec([(os.path.join(d, "wav.scp"), "speech", "sound")])
    # (e) what this path does not do is refused, not approximated
    with pytest.raises(NotImplementedError):
        CLI.inference_modelscope(dtype="float16", **common)
    with pytest.raises(NotImplementedError):
        CLI.inference_modelscope(ngpu=2, **common)
    fwd2 = CLI.inference_modelscope(output_dir=None, **common)
    with pytest.raises(ValueError):
        fwd2()
    # (e2) file_sampling_rate != sampling_rate: resample in, resample out, trimmed to the input length at the FILE rate
    #      (codec_inference.py:271-274,319-323,353-357)
    import torchaudio
    half = cfg.sample_rate // 2
    x8 = clips["u0"][: 40 * 6 + 3]
    got = fwd2(raw_inputs=x8, param_dict=dict(file_sampling_rate=half))
    up = torchaudio.functional.resample(torch.from_numpy(x8).view(1, -1), orig_freq=half, new_freq=cfg.sample_rate)
    rec = ora.inference(up, need_recon=True, bit_width=bw_all)["recon_speech"]
    want = torchaudio.functional.resample(rec, orig_freq=cfg.sample_rate, new_freq=half)[0][:, : x8.shape[0]]
    assert tuple(got[0]["value"].shape) == (1, x8.shape[0]) and torch.equal(got[0]["value"], want)
    with pytest.raises(NotImplementedError):
        fwd2(raw_inputs=os.path.join(d, "u2.wav"))                       # kwargs still carry file_sampling_rate = half
    with pytest.raises(NotImplementedError):
        CLI.inference_modelscope(output_dir=None, run_mod="decode", file_sampling_rate=half, **common)(raw_inputs=arr)
    # (f) inference(): positional mirror of the reference function, runs the pipeline once
    out2 = os.path.join(d, "out_inf")
    assert CLI.inference(out2, 2, "float32", 1, 0, 0, "INFO", [(os.path.join(d, "wav.scp"), "speech", "sound")],
                         os.path.join(d, "logdir", "keys.2.scp"), None, None, None, sampling_rate=cfg.sample_rate,
                         bit_width=bw_all, speech2token=s2t, run_mod="encode", need_indices=True) == []
    assert os.listdir(out2) == ["codecs.txt"]
    assert [l.split(" ", 1)[0] for l in open(os.path.join(out2, "codecs.txt"))] == ["u2"]


@pytest.mark.gpu
def test_cli_main_runs_the_scripts_three_stages(tmp_path):
    """`python -m funcodec_b200.bin.codec_inference` with encoding_decoding.sh's literal argument lists (stages 1-3, two JOBs):
    YAML + model.pth in, codecs.txt / wavs out, codes equal to the direct library call on the same wrap-padded batch."""
    from funcodec_b200.encodec import B200Encodec
    from funcodec_b200.speech2token import Speech2Token
    cfg = get_config("tiny_ds40")
    sd = init_state_dict(cfg, 3)
    d = str(tmp_path)
    os.makedirs(os.path.join(d, "model"))
    _yaml_for(cfg, os.path.join(d, "model"))
    torch.save(sd, os.path.join(d, "model", "model.pth"))
    lens = [40 * 9 + 5, 40 * 14, 40 * 6 + 39, 40 * 11]
    clips = _write_corpus(d, cfg, lens)
    for job in (1, 2):
        assert CLI.main(stage_argv(1, d, job=job, batch_size=2, sr=cfg.sample_rate)) == 2
    lines = []
    for job in (1, 2):
        lines += open(os.path.join(d, "logdir", f"output.{job}", "codecs.txt")).read().strip().split("\n")
    with open(os.path.join(d, "codecs.txt"), "wt") as f:
        f.write("\n".join(lines) + "\n")
    model = B200Encodec(cfg, sd, "cuda:0")
    n_q = min(cfg.num_quantizers_for_bandwidth(16000), cfg.num_quantizers)
    speech, _ = P.wrap_pad_batch([clips["u0"], clips["u1"]])
    ref = model.inference(speech, need_recon=False, bit_width=16000)["code_indices"][0].cpu()
    for i in range(2):
        key, arr = P.parse_indices_line(lines[i])
        tf = -(-lens[i] // cfg.hop_length)
        assert key == f"u{i}" and arr.shape == (tf, n_q) and np.array_equal(arr, ref[:, i, :tf].numpy().T)
    # stage 2 writes to output.JOB again: use fresh log dirs like the script does for each stage
    for stage, src in ((2, "codecs.txt"), (3, "emb.scp")):
        sd_dir = os.path.join(d, f"s{stage}")
        os.makedirs(os.path.join(sd_dir, "logdir"))
        for fn in ("model", src):
            os.symlink(os.path.join(d, fn), os.path.join(sd_dir, fn))
        for job in (1, 2):
            os.symlink(os.path.join(d, "logdir", f"keys.{job}.scp"), os.path.join(sd_dir, "logdir", f"keys.{job}.scp"))
        if stage == 3:
            continue
        for job in (1, 2):
            assert CLI.main(stage_argv(2, sd_dir, job=job, batch_size=2, sr=cfg.sample_rate)) == 2
        y, sr = P.load_wav(os.path.join(sd_dir, "logdir", "output.2", "u3.wav"))
        assert sr == cfg.sample_rate and y.shape[0] == 11 * cfg.hop_length
    # stage 3 input: embeddings of u0 / u1 from the library, as a Kaldi scp
    with ArkScpWriter(os.path.join(d, "emb")) as w:
        for key in ("u0", "u1"):
            e = model.inference(torch.from_numpy(clips[key]).view(1, -1), need_recon=False)["code_embeddings"][0][0]
            w(key, e[0].cpu().numpy())
    s3 = os.path.join(d, "s3")
    assert CLI.main(stage_argv(3, s3, job=1, batch_size=2, sr=cfg.sample_rate)) == 2
    y, _ = P.load_wav(os.path.join(s3, "logdir", "output.1", "u1.wav"))
    ref = model.inference_decoding_emb(model.inference(torch.from_numpy(clips["u1"]).view(1, -1), need_recon=False)
                                       ["code_embeddings"][0][0])["recon_speech"][0, 0].cpu()
    ref = P.peak_limit(ref, True).numpy()
    assert y.shape[0] == 14 * cfg.hop_length and np.abs(y - ref).max() <= 2.0 / 32768
