"""Pin the CPU oracle (oracle/encodec_oracle.py) on STEREO audio against vectors produced by the UNMODIFIED reference Encodec
built with input_size 2 / decoder_conf.channels 2 (tools/gen_golden_stereo.py -> tests/golden/model_stereo_small.npz): the RMS
scale of the mono mix (codec_basic.py:366-369), the 2-input first conv, the 2-output last conv with GroupNorm(1, 2) and
segmented overlap-add per channel.  CPU only; same pin as test_oracle_golden.py: equal codes, 2e-6 max-abs otherwise."""
import os

import numpy as np
import pytest
import torch

from funcodec_b200 import get_config, init_state_dict
from oracle import encodec_oracle as O

TOL = 2e-6
GOLDEN_THREADS = 8          # the thread count the vectors were generated with (see test_oracle_golden.py)


@pytest.fixture(autouse=True, scope="module")
def _golden_threads():
    n = torch.get_num_threads()
    torch.set_num_threads(GOLDEN_THREADS)
    yield
    torch.set_num_threads(n)


@pytest.fixture(scope="module")
def z(golden_dir):
    return np.load(os.path.join(golden_dir, "model_stereo_small.npz"))


def _model(z, pre, **kw):
    cfg = get_config(str(z[pre + "cfg_name"]))
    assert cfg.channels == 2
    sd = init_state_dict(cfg, int(z[pre + "seed"]))
    assert abs(sum(v.double().abs().sum().item() for v in sd.values()) - float(z[pre + "sd_checksum"])) <= \
        1e-6 * float(z[pre + "sd_checksum"]), "synthetic init drifted"
    assert tuple(sd["encoder.model.0.conv.conv." + ("weight_v" if cfg.norm == "weight_norm" else "weight")].shape)[:2] == (cfg.n_filters, 2)
    return cfg, sd, O.OracleEncodec.from_config(sd, cfg, **kw)


def _check_whole(z, pre, ora):
    wav = torch.from_numpy(z[pre + "wav"])
    B, C, L = wav.shape
    assert C == 2
    keys = sorted({k[len(pre):].split(".")[0] for k in z.files if k.startswith(pre) and k.endswith(".codes")})
    for key in keys:
        bw = None if key == "full" else int(key[2:])
        r = ora.inference(wav, need_recon=True, bit_width=bw, use_scale=True)
        assert np.array_equal(r["code_indices"][0].numpy(), z[f"{pre}{key}.codes"].astype(np.int64)), key
        assert np.abs(r["code_embeddings"][0][0].numpy() - z[f"{pre}{key}.quant"]).max() <= TOL
        assert np.abs(r["code_embeddings"][0][1].numpy() - z[f"{pre}{key}.scale"]).max() <= 1e-7
        assert r["recon_speech"].shape == z[f"{pre}{key}.recon"].shape == (B, 2, L)
        assert np.abs(r["recon_speech"].numpy() - z[f"{pre}{key}.recon"]).max() <= TOL, key
    r = ora.inference(wav)
    if pre + "encoder_out" in z.files:
        assert np.abs(r["encoder_out"].numpy() - z[pre + "encoder_out"]).max() <= TOL
        d = ora.inference_decoding(r["code_indices"][0].permute(1, 2, 0))
        assert np.abs(d["recon_speech"].numpy() - z[pre + "decode_codes.recon"]).max() <= TOL
        d = ora.inference_decoding_emb(r["code_embeddings"][0][0])
        assert np.abs(d["recon_speech"].numpy() - z[pre + "decode_emb.recon"]).max() <= TOL
        r2 = ora.inference(wav, use_scale=False)
        assert np.abs(r2["recon_speech"].numpy() - z[pre + "noscale.recon"]).max() <= TOL
    return r


def test_stereo_time_group_norm_lstm(z):
    _, _, ora = _model(z, "a.")
    r = _check_whole(z, "a.", ora)
    wav = torch.from_numpy(z["a.wav"])
    # the scale is the RMS of the mono mix, one value per clip
    mono = (wav[:, 0] + wav[:, 1]) * 0.5
    want = 1e-8 + mono.double().pow(2).mean(dim=-1).sqrt()
    assert np.allclose(r["code_embeddings"][0][1].view(-1).double().numpy(), want.numpy(), rtol=1e-6)
    # the two output channels are different signals (the C_out = 2 conv is not a copy of one channel)
    assert (r["recon_speech"][:, 0] - r["recon_speech"][:, 1]).abs().max() > 1e-3


def test_stereo_tiny_clip(z):
    """Clips shorter than one hop: the deep convs take pad1d's zero-extend-then-reflect branch (conv.py:89-97)."""
    _, _, ora = _model(z, "a.")
    _check_whole(z, "tiny.", ora)


def test_stereo_weight_norm_causal(z):
    """weight_norm + causal: the last conv has no GroupNorm, the stereo output is the plain conv output times the scale."""
    _, sd, ora = _model(z, "wn.")
    assert "decoder.model.0.conv.norm.weight" not in sd
    _check_whole(z, "wn.", ora)


def test_stereo_segmented(z):
    cfg, sd, _ = _model(z, "a.")
    dur, ov, B, L, seg, stride, n_seg = z["seg.meta"]
    ora = O.OracleEncodec.from_config(sd, cfg, segment_dur=float(dur), overlap_ratio=float(ov))
    assert O.segment_plan(int(L), cfg.sample_rate, float(dur), float(ov))[:2] == (int(seg), int(stride))
    r = ora.inference(torch.from_numpy(z["seg.wav"]))
    assert len(r["code_indices"]) == int(n_seg)
    for i in range(int(n_seg)):
        assert np.array_equal(r["code_indices"][i].numpy(), z[f"seg.codes{i}"].astype(np.int64))
        assert np.abs(r["code_embeddings"][i][0].numpy() - z[f"seg.quant{i}"]).max() <= TOL
        assert np.abs(r["code_embeddings"][i][1].numpy() - z[f"seg.scale{i}"]).max() <= 1e-7
    assert r["recon_speech"].shape == z["seg.recon"].shape == (int(B), 2, int(L))
    assert np.abs(r["recon_speech"].numpy() - z["seg.recon"]).max() <= TOL
