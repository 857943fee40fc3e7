"""Glue for the drop-in (INTEGRATION.md §3a): derive a CodecConfig from an already-built reference `Encodec`
(funcodec/models/codec_basic.py:119) or mag_phase `FreqCodec` (funcodec/models/codec_basic.py FreqCodec) module and wrap it with the CUDA-backed B200Encodec.

Only the configurations of DESIGN.md §9 are accepted; anything else raises (no silent fallback to the PyTorch path).
"""
from typing import Dict

import torch

from .config import CodecConfig


class UnsupportedReferenceModel(ValueError):
    pass


def config_from_reference_model(model) -> CodecConfig:
    """Reads the attributes SEANetEncoder / SEANetDecoder / CostumeQuantizer / Encodec keep
    (seanet_encoder.py:98-106, seanet_decoder.py:100-106, costume_quantizer.py:49-53, codec_basic.py:249-254)."""
    enc, dec, q = model.encoder, model.decoder, model.quantizer
    domain = getattr(model, "codec_domain", "time")
    freq = isinstance(domain, (list, tuple)) and list(domain) == ["mag_phase", "mag_phase"]
    if freq:        # FreqCodec (codec_freq.py): ratios are [freq, time] pairs
        pairs = [tuple(int(v) for v in r) for r in dec.ratios]
        if list(reversed(pairs)) != [tuple(int(v) for v in r) for r in enc.ratios]:
            raise UnsupportedReferenceModel("encoder/decoder ratios differ")
        ratios = tuple(p[1] for p in pairs)
        ratios_f = tuple(p[0] for p in pairs)
    else:
        if domain not in ("time", None) and not (isinstance(domain, (list, tuple)) and list(domain) == ["time", "time"]):
            raise UnsupportedReferenceModel(f"codec_domain {domain} is not supported (time, or ['mag_phase', 'mag_phase'])")
        ratios = tuple(int(r) for r in dec.ratios)
        ratios_f = ()
        if tuple(reversed(ratios)) != tuple(int(r) for r in enc.ratios):
            raise UnsupportedReferenceModel("encoder/decoder ratios differ")
    sd: Dict[str, torch.Tensor] = model.state_dict()
    # encoder_conf / decoder_conf `norm` (conv.py:21-55): weight_norm leaves weight_g / weight_v and no norm module,
    # time_group_norm a GroupNorm(1, C) per conv, none neither; spectral_norm / layer_norm are not built
    if any(k.endswith("weight_orig") or k.endswith("weight_u") for k in sd):
        raise UnsupportedReferenceModel("norm spectral_norm is not supported (time_group_norm, weight_norm or none)")
    wn = [k.endswith("weight_g") for k in sd if k.startswith(("encoder.model.", "decoder.model.")) and
          (k.endswith("conv.weight_g") or k.endswith("conv.weight") or k.endswith("convtr.weight_g") or k.endswith("convtr.weight"))]
    if any(wn) and not all(wn):
        raise UnsupportedReferenceModel("encoder and decoder must use the same norm")
    if any(wn):
        norm = "weight_norm"
    elif "encoder.model.0.conv.norm.weight" in sd:
        norm = "time_group_norm"
    else:
        norm = "none"
    if (norm == "time_group_norm") != ("decoder.model.0.conv.norm.weight" in sd):
        raise UnsupportedReferenceModel("encoder and decoder must use the same norm")
    if freq and norm != "time_group_norm":
        raise UnsupportedReferenceModel("FreqCodec: norm must be time_group_norm")
    if getattr(model, "segment_dur", None) is not None and freq:
        raise UnsupportedReferenceModel("segment_dur must be null for FreqCodec (whole-utterance processing)")
    if getattr(q, "input_proj", None) is not None or getattr(q, "input_act", None) is not None:
        raise UnsupportedReferenceModel("quantizer projections / codec_range are not supported")
    causal = _check_module_options(model)
    if causal and (freq or norm == "time_group_norm"):
        raise UnsupportedReferenceModel("causal convolutions need the time-domain stacks with norm weight_norm / none")
    embed = stacked_codebooks(sd)
    if embed is None:
        raise UnsupportedReferenceModel("no codebook buffers found (quantizer.rq.model.embed or ...layers.N._codebook.embed)")
    wk = "weight_v" if norm == "weight_norm" else "weight"
    w0 = sd["encoder.model.0.conv.conv." + wk]
    n_lstm = len([k for k in sd if k.startswith("decoder.model.1.lstm.weight_ih_l")])
    last_idx = max(int(k.split(".")[2]) for k in sd if k.startswith("decoder.model."))
    rb_k = sd["encoder.model.1.block.1.conv.conv." + wk].shape[-1]
    # stacked residual blocks (n_residual_layers): consecutive encoder.model.N with a shortcut conv; their first convs carry the
    # dilations dilation_base ** j (seanet_encoder.py:122-128)
    n_res = 1
    while f"encoder.model.{1 + n_res}.shortcut.conv.conv.{wk}" in sd:
        n_res += 1
    dil_base = 2
    if n_res > 1 and not freq and hasattr(enc, "model"):
        dils = []
        for j in range(n_res):
            blk = enc.model[1 + j]
            conv = blk.block[1].conv.conv
            dils.append(int(conv.dilation[0]))
        dil_base = dils[1] if dils[0] == 1 else 0
        if dil_base < 1 or any(dils[j] != dil_base ** j for j in range(n_res)):
            raise UnsupportedReferenceModel(f"residual-block dilations {dils} are not dilation_base ** j")
    if n_res > 1 and freq:
        raise UnsupportedReferenceModel("n_residual_layers > 1 is only supported for the time-domain stacks")
    # audio channels: SEANetEncoder.channels = input_size, SEANetDecoder.channels (seanet_encoder.py:98, seanet_decoder.py:101)
    channels = int(getattr(enc, "channels", 1) or 1) if not freq else 1
    if not freq and channels != int(getattr(dec, "channels", 1) or 1):
        raise UnsupportedReferenceModel(f"encoder channels {channels} != decoder channels {getattr(dec, 'channels', 1)}")
    if channels not in (1, 2):
        raise UnsupportedReferenceModel(f"{channels} audio channels: mono or stereo only (codec_basic.py:342-344)")
    dconf = getattr(model, "domain_conf", None) or {}
    cfg = CodecConfig(name="from_reference", ratios=ratios, arch=1 if freq else 0, ratios_f=ratios_f,
                      n_fft=int(dconf.get("n_fft", 512)), stft_hop=int(dconf.get("hop_length", 160)),
                      n_filters=int(w0.shape[0]), dimension=int(embed.shape[2]),
                      kernel_size=int(w0.shape[-1]),
                      last_kernel_size=int(sd[f"decoder.model.{last_idx}.conv.conv.{wk}"].shape[-1]),
                      residual_kernel_size=int(rb_k), lstm_layers=n_lstm, codebook_size=int(embed.shape[1]),
                      num_quantizers=int(embed.shape[0]), sample_rate=int(q.sampling_rate),
                      audio_normalize=bool(model.audio_normalize), n_residual_layers=n_res, dilation_base=dil_base,
                      norm=norm, causal=causal, channels=channels)
    if cfg.hop_length != int(q.encoder_hop_length):
        raise UnsupportedReferenceModel("quantizer.encoder_hop_length does not match prod(ratios)")
    if freq:
        # the modules do not keep conv_group_ratio / tr_conv_group_ratio: recover them from the weight shapes
        from dataclasses import replace
        from .weights import state_dict_shapes
        for gr in (-1, 1, 2, 4, 8, 16, 32):
            for tgr in (-1, 1, 2, 4, 8, 16, 32):
                cand = replace(cfg, conv_group_ratio=gr, tr_conv_group_ratio=tgr)
                try:
                    shapes = state_dict_shapes(cand)
                except ZeroDivisionError:
                    continue
                if all(tuple(sd[k].shape) == tuple(v) for k, v in shapes.items() if k in sd and k.endswith(".weight")):
                    return cand
        raise UnsupportedReferenceModel("2-D conv weight shapes match no conv_group_ratio / tr_conv_group_ratio")
    return cfg


def stacked_codebooks(sd):
    """[n_q, K, D] codebooks of either RVQ flavour: the stacked buffer of `use_ddp: true`
    (ddp_core_vq.py:349-352) or the per-layer buffers of `use_ddp: false` (core_vq.py:147-150) -- same semantics."""
    if "quantizer.rq.model.embed" in sd:
        return sd["quantizer.rq.model.embed"]
    per = []
    while f"quantizer.rq.model.layers.{len(per)}._codebook.embed" in sd:
        per.append(sd[f"quantizer.rq.model.layers.{len(per)}._codebook.embed"])
    return torch.stack(per, dim=0) if per else None


def _check_module_options(model) -> bool:
    """Options that change the maths but not the parameter names / shapes: inspect the module attributes
    (conv.py:240-241,275-276; lstm.py:19; ddp_core_vq.py:354-356; seanet_encoder.py:49-61) and refuse anything the engine does
    not build.  Returns the stacks' `causal` flag (one value for every conv of both stacks)."""
    import torch.nn as nn
    causal_seen = set()
    for side in ("encoder", "decoder"):
        net = getattr(model, side)
        if not hasattr(net, "modules"):       # not an nn.Module (a plain description object): nothing to inspect
            continue
        for mod in net.modules():
            name = type(mod).__name__
            if name in ("SConv1d", "SConv2d", "SConvTranspose1d", "SConvTranspose2d"):
                causal_seen.add(bool(getattr(mod, "causal", False)))
                if float(getattr(mod, "trim_right_ratio", 1.0)) != 1.0:
                    raise UnsupportedReferenceModel(f"{side}: trim_right_ratio must be 1")
                if getattr(mod, "pad_mode", "reflect") != "reflect":
                    raise UnsupportedReferenceModel(f"{side}: pad_mode must be reflect")
                norm_conv = getattr(mod, "conv", None) if hasattr(mod, "conv") else getattr(mod, "convtr", None)
                inner = getattr(norm_conv, "conv", None) if hasattr(norm_conv, "conv") else getattr(norm_conv, "convtr", None)
                nm = getattr(norm_conv, "norm", None)
                if nm is not None and type(nm).__name__ not in ("GroupNorm", "Identity"):
                    raise UnsupportedReferenceModel(f"{side}: norm module {type(nm).__name__} is not supported")
                if isinstance(nm, nn.GroupNorm) and int(nm.num_groups) != 1:
                    raise UnsupportedReferenceModel(f"{side}: GroupNorm must have one group (time_group_norm)")
                dil = getattr(inner, "dilation", (1,))
                if name != "SConv1d" and any(int(d) != 1 for d in dil):
                    raise UnsupportedReferenceModel(f"{side}: dilated 2-D / transposed convolutions are not supported")
            elif name == "SLSTM" and not getattr(mod, "skip", True):
                raise UnsupportedReferenceModel(f"{side}: SLSTM must use the skip connection (res_seq: true)")
            elif name in ("Snake1d", "Snake", "PReLU", "ReLU", "LeakyReLU", "GELU", "Tanh") or \
                    (isinstance(mod, nn.ELU) and float(mod.alpha) != 1.0):
                raise UnsupportedReferenceModel(f"{side}: activation must be ELU(alpha=1)")
    rq = getattr(getattr(model.quantizer, "rq", None), "model", None)
    if rq is not None and int(getattr(rq, "q0_ds_ratio", 1)) != 1:
        raise UnsupportedReferenceModel("quantizer q0_ds_ratio must be 1")
    if len(causal_seen) > 1:
        raise UnsupportedReferenceModel("encoder and decoder must agree on `causal`")
    return bool(causal_seen.pop()) if causal_seen else False


def wrap_reference_encodec(model, device: str = "cuda:0"):
    from .encodec import B200Encodec
    cfg = config_from_reference_model(model)
    return B200Encodec(cfg, model.state_dict(), device, segment_dur=getattr(model, "segment_dur", None),
                       overlap_ratio=getattr(model, "overlap_ratio", None))
