"""Generate tests/golden/model_stereo_small.npz: the UNMODIFIED reference Encodec (imported through tools/ref_harness.py)
built with input_size 2 and decoder_conf.channels 2 (seanet_encoder.py:63-65 names this stereo layout) at small widths, weights from
funcodec_b200.weights.init_state_dict loaded with load_state_dict.  Build container only:  python tools/gen_golden_stereo.py

Cases (key prefix):
  a.     stereo_small (time_group_norm, SLSTM): 3 ragged clips whose channels differ (one clip with the right channel a scaled
         copy of the left, one with a silent right channel), full n_q and one bandwidth limit, use_scale=False, encoder output,
         decode from codes and from embeddings
  tiny.  stereo_small on 2 clips shorter than one hop: the deep convs take pad1d's short-input branch (conv.py:89-97)
  seg.   stereo_small with segment_dur / overlap_ratio set: full segments and a short tail, linear overlap-add
  wn.    stereo_causal_small (weight_norm, causal, 3 dilated residual blocks, no LSTM): no GroupNorm on the last layer
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.dirname(HERE))

from ref_harness import build_reference_encodec  # noqa: E402
from funcodec_b200 import get_config, init_state_dict  # noqa: E402

OUT = os.path.join(os.path.dirname(HERE), "tests", "golden")
SEG = (0.01, 0.3)          # segment_dur 160 samples (4 frames of hop 40), stride 112


def sd_checksum(sd):
    return float(sum(v.double().abs().sum().item() for v in sd.values()))


def stereo_wav(B, L, seed):
    g = torch.Generator().manual_seed(seed)
    wav = 0.1 * torch.randn(B, 2, L, generator=g)
    if B >= 3:
        wav[1, 1] = 0.5 * wav[1, 0]           # right = scaled left
        wav[2, 1] = 0.0                       # silent right channel
    return wav


def whole_case(out, pre, model, wav, bit_widths=(None,)):
    out[pre + "wav"] = wav.numpy()
    with torch.no_grad():
        for bw in bit_widths:
            key = pre + ("full" if bw is None else f"bw{bw}")
            r = model.inference(wav, need_recon=True, bit_width=bw, use_scale=True)
            out[key + ".codes"] = r["code_indices"][0].numpy().astype(np.int16)
            out[key + ".quant"] = r["code_embeddings"][0][0].numpy()
            out[key + ".scale"] = r["code_embeddings"][0][1].numpy()
            out[key + ".recon"] = r["recon_speech"].numpy()
            if bw is None:
                emb, _ = model._encode(wav)[0]
                out[pre + "encoder_out"] = emb.numpy()
                toks = r["code_indices"][0].permute(1, 2, 0)
                out[pre + "decode_codes.recon"] = model.inference_decoding(toks)["recon_speech"].numpy()
                out[pre + "decode_emb.recon"] = model.inference_decoding_emb(r["code_embeddings"][0][0])["recon_speech"].numpy()
                out[pre + "noscale.recon"] = model.inference(wav, need_recon=True, bit_width=None, use_scale=False)["recon_speech"].numpy()


def main():
    torch.set_num_threads(8)
    out = {}
    for pre, name, seed in (("a.", "stereo_small", 0), ("wn.", "stereo_causal_small", 3)):
        cfg = get_config(name)
        sd = init_state_dict(cfg, seed)
        out[pre + "cfg_name"] = name
        out[pre + "seed"] = seed
        out[pre + "sd_checksum"] = sd_checksum(sd)
        model = build_reference_encodec(cfg)
        model.load_state_dict(sd)
        if pre == "a.":
            whole_case(out, pre, model, stereo_wav(3, 40 * 23 + 17, 21), bit_widths=(None, 8000))
            whole_case(out, "tiny.", model, stereo_wav(2, 29, 22))
            dur, ov = SEG
            model.segment_dur, model.overlap_ratio = dur, ov
            wav = stereo_wav(2, 620, 23)
            with torch.no_grad():
                r = model.inference(wav, need_recon=True, bit_width=None, use_scale=True)
            out["seg.meta"] = np.array([dur, ov, 2, 620, model.segment_length, model.segment_stride, len(r["code_indices"])])
            out["seg.wav"] = wav.numpy()
            out["seg.recon"] = r["recon_speech"].numpy()
            for i, (codes, (quant, scale)) in enumerate(zip(r["code_indices"], r["code_embeddings"])):
                out[f"seg.codes{i}"] = codes.numpy().astype(np.int16)
                out[f"seg.quant{i}"] = quant.numpy()
                out[f"seg.scale{i}"] = scale.numpy()
            print("seg: segments", [tuple(c.shape) for c in r["code_indices"]], tuple(r["recon_speech"].shape))
            model.segment_dur, model.overlap_ratio = None, None
        else:
            whole_case(out, pre, model, stereo_wav(2, 40 * 21 + 9, 24))
    path = os.path.join(OUT, "model_stereo_small.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path) // 1024, "KiB")


if __name__ == "__main__":
    main()
