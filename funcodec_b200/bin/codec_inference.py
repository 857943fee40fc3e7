"""Drop-in for `python -m funcodec.bin.codec_inference` (funcodec/bin/codec_inference.py:428-575) backed by the CUDA library:
the same flag set, so the command lines of `egs/LibriTTS/codec/encoding_decoding.sh:80-98,124-143,168-187` (stages 1-3) run
unchanged with the module path swapped:

    python -m funcodec_b200.bin.codec_inference --batch_size 16 --num_workers 4 --ngpu 1 --gpuid_list 0,1 \
        --data_path_and_name_and_type wav.scp,speech,sound --key_file logdir/keys.1.scp \
        --config_file exp/model/config.yaml --model_file exp/model/model.pth --output_dir logdir/output.1 \
        --sampling_rate 16000 --file_sampling_rate 16000 --bit_width 16000 --need_indices true --need_sub_quants false \
        --use_scale false --indices_save_type text --run_mod encode

`config.yaml` is the training config the reference saves (encoder_conf / quantizer_conf / decoder_conf / model_conf, time-domain
Encodec or mag_phase FreqCodec); `model.pth` is the plain state_dict.  Unsupported configurations are refused loudly (no fallback
to a PyTorch path).  Defaults equal the reference parser's (`--use_scale true`, `--bit_width 16000`, `--batch_size 1`).
"""
import argparse
import math
import os
import sys

import numpy as np
import torch
import yaml

from funcodec_b200.config import CodecConfig
from funcodec_b200.encodec import B200Encodec
from funcodec_b200.pipeline import forward_items, load_items, run_decode, run_decode_emb, run_encode
from funcodec_b200.speech2token import Speech2Token


def str2bool(v: str) -> bool:
    """funcodec.utils.types.str2bool."""
    if v.lower() in ("true", "1", "yes", "y", "t"):
        return True
    if v.lower() in ("false", "0", "no", "n", "f"):
        return False
    raise argparse.ArgumentTypeError(f"not a boolean: {v}")


def str_or_none(v: str):
    return None if v.lower() in ("none", "null", "nil", "") else v


def str2triple_str(v: str):
    parts = [x.strip() for x in v.strip().strip("()[]").split(",")]
    if len(parts) != 3:
        raise argparse.ArgumentTypeError(f"expected path,name,type: {v}")
    return tuple(parts)


def config_from_yaml(path: str):
    """-> (CodecConfig, segment_dur, overlap_ratio) from the reference's training YAML
    (egs/LibriTTS/codec/conf/*.yaml; gan_speech_codec.py:301-358 feeds these dicts to the model classes)."""
    with open(path, "rt", encoding="utf-8") as f:
        a = yaml.safe_load(f)
    enc, dec, q, m = a.get("encoder_conf", {}), a.get("decoder_conf", {}), a.get("quantizer_conf", {}), a.get("model_conf", {})

    def refuse(msg):
        raise SystemExit(f"unsupported configuration: {msg}")

    for side, conf in (("encoder_conf", enc), ("decoder_conf", dec)):
        # the classes default to norm='weight_norm', causal=False (seanet_encoder.py:93-94, seanet_decoder.py:92-93)
        if conf.get("norm", "weight_norm") not in ("time_group_norm", "weight_norm", "none"):
            refuse(f"{side}.norm must be time_group_norm, weight_norm or none")
        if conf.get("causal", False) and conf.get("norm", "weight_norm") == "time_group_norm":
            refuse(f"{side}: GroupNorm doesn't support causal evaluation (conv.py:46-47)")
        if float(conf.get("trim_right_ratio", 1.0)) != 1.0:
            refuse(f"{side}.trim_right_ratio must be 1")
        if conf.get("seq_model", "lstm") not in ("lstm", "none", None):
            refuse(f"{side}.seq_model must be lstm or none")
        if conf.get("activation", "ELU") != "ELU" or conf.get("pad_mode", "reflect") != "reflect":
            refuse(f"{side}: activation must be ELU and pad_mode reflect")
    if q.get("codec_dim") is not None or q.get("codec_range") is not None:
        refuse("quantizer projections / codec_range")
    if int(q.get("q0_ds_ratio", 1) or 1) != 1:
        refuse("quantizer_conf.q0_ds_ratio must be 1")
    if enc.get("norm", "weight_norm") != dec.get("norm", "weight_norm") or bool(enc.get("causal", False)) != bool(dec.get("causal", False)):
        refuse("encoder_conf and decoder_conf must agree on norm and causal")
    for key in ("n_residual_layers", "dilation_base", "seq_model"):
        if enc.get(key, None) != dec.get(key, None):
            refuse(f"encoder_conf.{key} != decoder_conf.{key}")
    ratios = dec.get("ratios", [8, 5, 4, 2])
    if enc.get("ratios", [8, 5, 4, 2]) != ratios:
        refuse("encoder and decoder ratios differ")
    domain = m.get("codec_domain", None)
    # audio channels: top-level input_size feeds SEANetEncoder(input_size=...) and decoder_conf.channels the decoder's last
    # conv (gan_speech_codec.py:304-329); the reference Encodec takes 1 or 2 (codec_basic.py:342-344)
    channels = int(a.get("input_size", 1) or 1)
    kw = {}
    if a.get("model", "encodec") == "freq_codec" or (ratios and isinstance(ratios[0], (list, tuple))):
        if list(domain or []) != ["mag_phase", "mag_phase"]:
            refuse("FreqCodec codec_domain must be ['mag_phase', 'mag_phase']")
        dconf = m.get("domain_conf", {}) or {}
        kw = dict(arch=1, ratios_f=tuple(int(r[0]) for r in ratios), n_fft=int(dconf.get("n_fft", 512)),
                  stft_hop=int(dconf.get("hop_length", 160)), conv_group_ratio=int(enc.get("conv_group_ratio", -1)),
                  tr_conv_group_ratio=int(dec.get("tr_conv_group_ratio", -1)))
        if int(dec.get("conv_group_ratio", enc.get("conv_group_ratio", -1))) != kw["conv_group_ratio"]:
            refuse("encoder / decoder conv_group_ratio differ")
        ratios = [int(r[1]) for r in ratios]
        if m.get("segment_dur") is not None:
            refuse("segment_dur must be null for FreqCodec")
        if enc.get("norm", "weight_norm") != "time_group_norm" or enc.get("causal", False):
            refuse("FreqCodec: norm must be time_group_norm and causal false")
        channels = 1          # input_size there counts the spectral features of the 2-D stacks; the waveform is mono
    elif domain not in (None, "time", ["time", "time"]):
        refuse(f"codec_domain {domain}")
    else:
        if int(dec.get("channels", 1)) != channels:
            refuse(f"input_size {channels} != decoder_conf.channels {dec.get('channels', 1)}")
        if channels not in (1, 2):
            refuse(f"input_size {channels}: mono or stereo only")
    cfg = CodecConfig(name="from_yaml", ratios=tuple(int(r) for r in ratios), n_filters=int(enc.get("n_filters", 32)),
                      dimension=int(m.get("odim", 128)), kernel_size=int(enc.get("kernel_size", 7)),
                      last_kernel_size=int(enc.get("last_kernel_size", 7)),
                      residual_kernel_size=int(enc.get("residual_kernel_size", 3)),
                      codebook_size=int(q.get("codebook_size", 1024)), num_quantizers=int(q.get("num_quantizers", 32)),
                      sample_rate=int(q.get("sampling_rate", 16000)), audio_normalize=bool(m.get("audio_normalize", True)),
                      lstm_layers=int(enc.get("seq_layer_num", 2)) if enc.get("seq_model", "lstm") == "lstm" else 0,
                      n_residual_layers=int(enc.get("n_residual_layers", 1)),
                      # with one residual block the dilation base never shows (base ** 0 == 1): keep the default so that equal
                      # models compare equal
                      dilation_base=int(enc.get("dilation_base", 2)) if int(enc.get("n_residual_layers", 1)) > 1 else 2,
                      norm=str(enc.get("norm", "weight_norm")), causal=bool(enc.get("causal", False)), channels=channels, **kw)
    if int(q.get("encoder_hop_length", cfg.hop_length)) != cfg.hop_length:
        refuse("quantizer_conf.encoder_hop_length != hop of the ratios")
    return cfg, m.get("segment_dur"), m.get("overlap_ratio")


def get_parser():
    """Same flags, types and defaults as the reference's get_parser (codec_inference.py:428-558)."""
    p = argparse.ArgumentParser(description="Speech Tokenizer (B200)", formatter_class=argparse.ArgumentDefaultsHelpFormatter)
    p.add_argument("--log_level", type=lambda x: x.upper(), default="INFO",
                   choices=("CRITICAL", "ERROR", "WARNING", "INFO", "DEBUG", "NOTSET"))
    p.add_argument("--output_dir", type=str, required=False)
    p.add_argument("--ngpu", type=int, default=0, help="accepted for compatibility; this implementation always runs on a GPU")
    p.add_argument("--gpuid_list", type=str, default="")
    p.add_argument("--seed", type=int, default=0)
    p.add_argument("--dtype", default="float32", choices=["float16", "float32", "float64"])
    p.add_argument("--num_workers", type=int, default=0, help="accepted for compatibility (host I/O is in-process)")
    g = p.add_argument_group("Input data related")
    g.add_argument("--data_path_and_name_and_type", type=str2triple_str, required=False, action="append")
    g.add_argument("--key_file", type=str_or_none)
    g.add_argument("--allow_variable_data_keys", type=str2bool, default=False)
    g = p.add_argument_group("The model configuration related")
    g.add_argument("--config_file", type=str)
    g.add_argument("--model_file", type=str)
    g.add_argument("--model_tag", type=str)
    p.add_argument("--batch_size", type=int, default=1)
    p.add_argument("--sampling_rate", type=int, default=24_000)
    p.add_argument("--file_sampling_rate", type=int, default=None)
    p.add_argument("--bit_width", type=int, default=16_000)
    p.add_argument("--use_scale", type=str2bool, default=True)
    g.add_argument("--need_indices", type=str2bool)
    g.add_argument("--indices_save_type", type=str, default="text")
    g.add_argument("--need_sub_quants", type=str2bool)
    g.add_argument("--run_mod", type=str, choices=["inference", "encode", "decode", "decode_emb"], default="inference")
    g.add_argument("--stat_flops", type=str2bool, default=False)
    return p


def pick_gpu(output_dir, gpuid_list: str) -> int:
    """codec_inference.py:565-575: the job id is the suffix of `--output_dir` (`.../output.JOB`) and selects the GPU
    round-robin from `--gpuid_list`."""
    ids = [x for x in gpuid_list.split(",") if x != ""] or ["0"]
    jobid = 1
    if output_dir is not None:
        try:
            jobid = int(str(output_dir).split(".")[-1])
        except ValueError:
            jobid = 1
    return int(ids[(jobid - 1) % len(ids)])


def stat_flops_line(cfg: CodecConfig, bit_width=None) -> str:
    """`--stat_flops` (codec_inference.py:329-345 profiles the torch modules with thop on ONE SECOND of audio and logs parameters
    and MACs): the same two totals from the analytic model of this path (funcodec_b200/workload.py), per second of audio."""
    from funcodec_b200.workload import workload_model
    n_q = min(cfg.num_quantizers_for_bandwidth(bit_width), cfg.num_quantizers) if bit_width else cfg.num_quantizers
    w = workload_model(cfg, cfg.sample_rate, n_q=n_q)
    n_par = w["conv_params"] + w["lstm_params"] + w["codebook_params"]
    return (f"Model parameters: {n_par / 1e6:.2f}M, model flops: {w['total_macs'] / 1e9:.2f}G MACs per second of audio "
            f"(conv {w['conv_macs'] / 1e9:.2f}G, LSTM {w['lstm_macs'] / 1e9:.2f}G, RVQ@{n_q} {w['rvq_flops'] / 2e9:.2f}G)")


def refuse_stereo_file_io(cfg: CodecConfig):
    """The file I/O here (wav.scp / PCM16 wav, one channel per utterance) is mono; the reference CLI cannot feed a stereo model
    either (its [B, L, C] batches fail _encode's channel assert).  Stereo models run through B200Encodec with [B, 2, L] tensors."""
    if cfg.channels != 1:
        raise SystemExit(f"unsupported configuration: input_size {cfg.channels} (stereo) through the CLI's mono file I/O; "
                         "call funcodec_b200.B200Encodec.inference with [B, 2, L] tensors instead")


def build_speech2token(config_file: str, model_file: str, device: str = "cuda:0", need_sub_quants: bool = False):
    """`Speech2Token.from_pretrained` without the hub (codec_inference.py:136-150): YAML + checkpoint -> Speech2Token on B200Encodec."""
    cfg, segment_dur, overlap_ratio = config_from_yaml(config_file)
    refuse_stereo_file_io(cfg)
    sd = torch.load(model_file, map_location="cpu")
    if isinstance(sd, dict) and "state_dict" in sd and not any(k.startswith("encoder.") for k in sd):
        sd = sd["state_dict"]
    model = B200Encodec(cfg, sd, device, segment_dur=segment_dur, overlap_ratio=overlap_ratio)
    return Speech2Token(model, device, need_sub_quants=need_sub_quants)


def inference_modelscope(output_dir=None, batch_size: int = 1, dtype: str = "float32", ngpu: int = 1, seed: int = 0,
                         num_workers: int = 0, log_level="INFO", key_file=None, config_file="config.yaml",
                         model_file="model.pth", model_tag=None, allow_variable_data_keys: bool = True, streaming: bool = False,
                         sampling_rate: int = 16_000, bit_width: int = 8_000, param_dict=None, use_scale=True, **kwargs):
    """The callable-pipeline entry the modelscope wrapper and `inference()` use (codec_inference.py:164-382): builds the model once
    and returns `_forward(data_path_and_name_and_type=None, raw_inputs=None, output_dir_v2=None, param_dict=None)`.  Same
    arguments, defaults and return convention: with an output directory the results go to files (wav, codecs.txt / indices.ark,
    codec_emb.ark per `need_indices` / `indices_save_type` / `need_sub_quants` in kwargs / param_dict) and the list is empty; without
    one, a list of {"key", "value": reconstructed wav [1, L]}.  `raw_inputs`: samples (ndarray / tensor) or a wav path, key "utt" /
    the file's basename.  `file_sampling_rate` != `sampling_rate` resamples like the reference (torchaudio, host side).  Not
    available here: `model_tag` (hub), `dtype` other than float32.  `stat_flops` logs the analytic counts (stat_flops_line).  Extra keyword for embedding / tests: `speech2token=` an already built Speech2Token-like callable,
    `device=` (default cuda:<--gpuid_list pick>)."""
    if param_dict is not None:
        kwargs.update(param_dict)
    if ngpu > 1:
        raise NotImplementedError("only single GPU decoding is supported")         # as the reference (codec_inference.py:190-191)
    if dtype != "float32":
        raise NotImplementedError("dtype: only float32 is implemented (fp32-parity kernels)")
    if model_tag:
        raise NotImplementedError("model_tag (model hub download) is not available; pass config_file / model_file")
    s2t = kwargs.pop("speech2token", None)
    device = kwargs.pop("device", None) or f"cuda:{pick_gpu(output_dir, kwargs.get('gpuid_list', '') or '')}"
    if s2t is None:
        s2t = build_speech2token(config_file, model_file, device, need_sub_quants=bool(kwargs.get("need_sub_quants")))
    model_rate = s2t.model.quantizer.sampling_rate
    if model_rate != sampling_rate:
        raise ValueError(f"sampling_rate {sampling_rate} != model rate {model_rate}")

    def _forward(data_path_and_name_and_type=None, raw_inputs=None, output_dir_v2=None, param_dict=None):
        if param_dict is not None:
            kwargs.update(param_dict)
        file_rate = kwargs.get("file_sampling_rate") or sampling_rate
        if kwargs.get("stat_flops") and getattr(s2t.model, "cfg", None) is not None and not getattr(s2t, "already_stat_flops", False):
            import logging
            logging.info(stat_flops_line(s2t.model.cfg, bit_width))
            s2t.already_stat_flops = True
        run_mod = kwargs.get("run_mod", "inference")
        if data_path_and_name_and_type is None and raw_inputs is not None:
            uttid = "utt"
            if isinstance(raw_inputs, str):
                uttid = os.path.basename(raw_inputs).rsplit(".")[0]
                from funcodec_b200.pipeline import load_wav
                if file_rate != sampling_rate:
                    # (the reference loads the file AT the model rate and then resamples it again by file_sampling_rate)
                    raise NotImplementedError("a wav path as raw_inputs together with file_sampling_rate != sampling_rate")
                raw_inputs, sr = load_wav(raw_inputs)       # the reference resamples the file to the model rate while loading
                if sr != sampling_rate:
                    import torchaudio
                    raw_inputs = torchaudio.functional.resample(torch.from_numpy(raw_inputs), orig_freq=sr, new_freq=sampling_rate)
            if isinstance(raw_inputs, torch.Tensor):
                raw_inputs = raw_inputs.numpy()
            items = [(uttid, np.asarray(raw_inputs))]
        elif data_path_and_name_and_type:
            path, _name, dtype_ = data_path_and_name_and_type[0]
            want = {"decode": ("codec_json", "text"), "decode_emb": ("kaldi_ark",)}.get(run_mod, ("sound",))
            if dtype_ not in want:
                raise ValueError(f"run_mod {run_mod} reads {want[0]}, got {dtype_}")
            items = load_items(path, dtype_, key_file)
        else:
            raise ValueError("need data_path_and_name_and_type or raw_inputs")
        bw = param_dict["bit_width"] if param_dict is not None and "bit_width" in param_dict else bit_width
        output_path = output_dir_v2 if output_dir_v2 is not None else output_dir
        return forward_items(s2t, items, output_path, batch_size=batch_size, bit_width=bw, use_scale=use_scale, run_mod=run_mod,
                             need_indices=bool(kwargs.get("need_indices")), indices_save_type=kwargs.get("indices_save_type", "text"),
                             need_sub_quants=bool(kwargs.get("need_sub_quants")), sample_rate=sampling_rate,
                             file_sample_rate=file_rate)

    return _forward


def inference(output_dir, batch_size, dtype, ngpu, seed, num_workers, log_level, data_path_and_name_and_type, key_file,
              config_file, model_file, model_tag, allow_variable_data_keys: bool = True, streaming: bool = False,
              sampling_rate: int = 24_000, bit_width: int = 24_000, use_scale: bool = True, **kwargs):
    """codec_inference.py:385-425: build the pipeline, run it once on the data files."""
    pipeline = inference_modelscope(output_dir=output_dir, batch_size=batch_size, dtype=dtype, ngpu=ngpu, seed=seed,
                                    num_workers=num_workers, log_level=log_level, key_file=key_file, config_file=config_file,
                                    model_file=model_file, model_tag=model_tag, allow_variable_data_keys=allow_variable_data_keys,
                                    streaming=streaming, sampling_rate=sampling_rate, bit_width=bit_width, use_scale=use_scale,
                                    **kwargs)
    return pipeline(data_path_and_name_and_type, raw_inputs=None)


def main(argv=None):
    args = get_parser().parse_args(argv)
    if args.file_sampling_rate is None:
        args.file_sampling_rate = args.sampling_rate
    if args.dtype != "float32":
        raise SystemExit("--dtype: only float32 is implemented (fp32-parity kernels)")
    if args.model_tag:
        raise SystemExit("--model_tag (model hub download) is not available; pass --config_file / --model_file")
    resample = args.file_sampling_rate != args.sampling_rate
    if resample and args.run_mod in ("decode", "decode_emb"):
        raise SystemExit("--file_sampling_rate != --sampling_rate is only defined for --run_mod inference / encode")
    if not args.data_path_and_name_and_type:
        raise SystemExit("--data_path_and_name_and_type is required")
    if args.output_dir is None:
        raise SystemExit("--output_dir is required (raw_inputs mode is a Python API: funcodec_b200.speech2token)")
    path, _name, dtype = args.data_path_and_name_and_type[0]
    device = f"cuda:{pick_gpu(args.output_dir, args.gpuid_list)}"
    cfg, segment_dur, overlap_ratio = config_from_yaml(args.config_file)
    refuse_stereo_file_io(cfg)
    if cfg.sample_rate != args.sampling_rate:
        raise SystemExit(f"--sampling_rate {args.sampling_rate} != model rate {cfg.sample_rate}")
    if args.stat_flops:
        print(stat_flops_line(cfg, args.bit_width), file=sys.stderr)
    sd = torch.load(args.model_file, map_location="cpu")
    if isinstance(sd, dict) and "state_dict" in sd and not any(k.startswith("encoder.") for k in sd):
        sd = sd["state_dict"]
    model = B200Encodec(cfg, sd, device, segment_dur=segment_dur, overlap_ratio=overlap_ratio)
    s2t = Speech2Token(model, device, need_sub_quants=bool(args.need_sub_quants))
    if args.run_mod == "decode":
        if dtype not in ("codec_json", "text"):
            raise SystemExit(f"--run_mod decode reads codec_json, got {dtype}")
        n = run_decode(s2t, path, args.output_dir, args.batch_size, args.bit_width, key_file=args.key_file)
    elif args.run_mod == "decode_emb":
        if dtype not in ("kaldi_ark",):
            raise SystemExit(f"--run_mod decode_emb reads kaldi_ark, got {dtype}")
        n = run_decode_emb(s2t, path, args.output_dir, args.batch_size, key_file=args.key_file)
    elif resample:
        # resampled I/O (codec_inference.py:271-274,319-323,353-357): the generic batch loop, which resamples where the reference does
        if dtype != "sound":
            raise SystemExit(f"--run_mod {args.run_mod} reads sound, got {dtype}")
        items = load_items(path, dtype, args.key_file)
        forward_items(s2t, items, args.output_dir, batch_size=args.batch_size, bit_width=args.bit_width, use_scale=args.use_scale,
                      run_mod=args.run_mod, need_indices=bool(args.need_indices), indices_save_type=args.indices_save_type,
                      need_sub_quants=bool(args.need_sub_quants), file_sample_rate=args.file_sampling_rate)
        n = len(items)
    else:
        if dtype != "sound":
            raise SystemExit(f"--run_mod {args.run_mod} reads sound, got {dtype}")
        n = run_encode(s2t, path, args.output_dir, args.batch_size, args.bit_width, args.run_mod, args.use_scale,
                       key_file=args.key_file, need_indices=bool(args.need_indices),
                       indices_save_type=args.indices_save_type, need_sub_quants=bool(args.need_sub_quants))
    print(f"processed {n} utterances -> {args.output_dir}", file=sys.stderr)
    return n


if __name__ == "__main__":
    main(sys.argv[1:])
