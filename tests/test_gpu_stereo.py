"""Stereo (two-channel) time-domain Encodec on the GPU, on both conv paths (use_tc 1 and 0): parity with the vectors of the
UNMODIFIED reference (tests/golden/model_stereo_small.npz, tools/gen_golden_stereo.py), the two stereo layers alone against a
float64 evaluation, the full-width encodec_48k_stereo preset against the oracle, and the properties of the scale and batch.

Bars as in test_gpu_parity.py: codes bit-exact up to margin-classified near-ties, waveforms 1e-4 max-abs on clips whose codes
all match and on the decode-only paths; layers 2e-5 x rms."""
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from funcodec_b200 import get_config, init_state_dict
from funcodec_b200._capi import FcbError
from oracle import encodec_oracle as O
from parity_utils import assert_codes_parity

pytestmark = pytest.mark.gpu

WAV_TOL = 1e-4
EMB_TOL = 5e-5
MARGIN_E2E = 2e-3
PATHS = pytest.mark.parametrize("use_tc", [1, 0], ids=["tc", "simt"])

_MODELS = {}


def _model(cfg_name, seed, use_tc=1, **kw):
    from funcodec_b200.encodec import B200Encodec
    key = (cfg_name, seed, use_tc, tuple(sorted(kw.items())))
    if key not in _MODELS:
        cfg = get_config(cfg_name)
        sd = init_state_dict(cfg, seed)
        _MODELS[key] = (cfg, sd, B200Encodec(cfg, sd, "cuda:0", options={"use_tc": use_tc}, **kw),
                        O.OracleEncodec.from_config(sd, cfg, **kw))
    return _MODELS[key]


def _np(t):
    return t.detach().cpu().numpy()


@pytest.fixture(scope="module")
def z(golden_dir):
    return np.load(os.path.join(golden_dir, "model_stereo_small.npz"))


def _check_whole(z, pre, model, oracle, what):
    wav = torch.from_numpy(z[pre + "wav"])
    B, C, L = wav.shape
    ora = oracle.inference(wav, want_margin=True)
    assert np.array_equal(_np(ora["code_indices"][0]), z[pre + "full.codes"].astype(np.int64)), "oracle != golden"
    keys = sorted({k[len(pre):].split(".")[0] for k in z.files if k.startswith(pre) and k.endswith(".codes")})
    for key in keys:
        bw = None if key == "full" else int(key[2:])
        ora_k = ora if bw is None else oracle.inference(wav, bit_width=bw, want_margin=True)
        r = model.inference(wav, need_recon=True, bit_width=bw, need_encoder_out=bw is None)
        codes = _np(r["code_indices"][0])
        res = assert_codes_parity(codes, z[f"{pre}{key}.codes"], _np(ora_k["margins"]), MARGIN_E2E, what=f"{what} {pre}{key}")
        scale = _np(r["code_embeddings"][0][1])
        assert np.abs(scale - z[f"{pre}{key}.scale"]).max() <= 1e-6 * np.abs(z[f"{pre}{key}.scale"]).max()
        recon, quant = _np(r["recon_speech"]), _np(r["code_embeddings"][0][0])
        assert recon.shape == z[f"{pre}{key}.recon"].shape == (B, 2, L)
        ok_clip = ~(res["first_stage"] >= 0).any(axis=1)
        for b in np.nonzero(ok_clip)[0]:
            assert np.abs(quant[b] - z[f"{pre}{key}.quant"][b]).max() <= 1e-5
            assert np.abs(recon[b] - z[f"{pre}{key}.recon"][b]).max() <= WAV_TOL, (key, b)
        if bw is None:
            enc = _np(r["encoder_out"])
            assert np.abs(enc - z[pre + "encoder_out"]).max() <= EMB_TOL
    # decode-only paths: same inputs in, no index contamination
    d = model.inference_decoding_emb(torch.from_numpy(z[pre + "full.quant"]))
    assert _np(d["recon_speech"]).shape == z[pre + "decode_emb.recon"].shape
    assert np.abs(_np(d["recon_speech"]) - z[pre + "decode_emb.recon"]).max() <= WAV_TOL
    toks = torch.from_numpy(z[pre + "full.codes"].astype(np.int64)).permute(1, 2, 0)
    d = model.inference_decoding(toks)
    assert np.abs(_np(d["recon_speech"]) - z[pre + "decode_codes.recon"]).max() <= WAV_TOL
    # use_scale=False
    if pre + "noscale.recon" in z.files:
        r = model.inference(wav, need_recon=True, use_scale=False)
        if np.array_equal(_np(r["code_indices"][0]), z[pre + "full.codes"].astype(np.int64)):
            assert np.abs(_np(r["recon_speech"]) - z[pre + "noscale.recon"]).max() <= WAV_TOL


@PATHS
@pytest.mark.parametrize("pre, name, seed", [("a.", "stereo_small", 0), ("tiny.", "stereo_small", 0),
                                             ("wn.", "stereo_causal_small", 3)])
def test_stereo_golden(z, pre, name, seed, use_tc):
    assert str(z[("a." if pre == "tiny." else pre) + "cfg_name"]) == name
    _, _, model, oracle = _model(name, seed, use_tc)
    _check_whole(z, pre, model, oracle, f"stereo {'tc' if use_tc else 'simt'}")


@PATHS
def test_stereo_golden_segmented(z, use_tc):
    dur, ov, B, L, seg, stride, n_seg = z["seg.meta"]
    _, _, model, oracle = _model("stereo_small", 0, use_tc, segment_dur=float(dur), overlap_ratio=float(ov))
    wav = torch.from_numpy(z["seg.wav"])
    ora = oracle.inference(wav, want_margin=True)
    r = model.inference(wav, need_recon=True)
    assert len(r["code_indices"]) == int(n_seg)
    all_ok = True
    for i in range(int(n_seg)):
        res = assert_codes_parity(_np(r["code_indices"][i]), z[f"seg.codes{i}"], _np(ora["margins"][i]), MARGIN_E2E,
                                  what=f"stereo segmented {i}")
        all_ok = all_ok and res["exact_frames"] == res["total_frames"]
        assert np.abs(_np(r["code_embeddings"][i][1]) - z[f"seg.scale{i}"]).max() <= 1e-6 * np.abs(z[f"seg.scale{i}"]).max()
    recon = _np(r["recon_speech"])
    assert recon.shape == z["seg.recon"].shape == (int(B), 2, int(L))
    if all_ok:
        assert np.abs(recon - z["seg.recon"]).max() <= WAV_TOL


# ------------------------------------------------------------------------------------------------ layer level
def _truth(x_bct, w, b, stride=1):
    x = x_bct.double()
    pl, pr = O.conv_paddings(x.shape[-1], w.shape[-1], stride, 1)
    return F.conv1d(O.pad1d_reflect(x, (pl, pr)), w.double(), b.double(), stride=stride)


@PATHS
@pytest.mark.parametrize("layer, T, elu", [("encoder.model.0", 4801, False), ("encoder.model.0", 3, False),
                                           ("decoder.model.15", 3000, True), ("decoder.model.15", 1500 + 7, True),
                                           ("decoder.model.15", 5, True)])
def test_stereo_layers(layer, T, elu, use_tc):
    """The C_in = 2 first conv (planar input) and the C_out = 2 last conv with its GroupNorm(1, 2) statistics, through
    fcb_debug_conv1d on the full-width stereo preset (C_in = 32: the templated small-C_out kernel), against float64."""
    cfg, sd, model, _ = _model("encodec_48k_stereo", 0, use_tc)
    cin = 2 if layer == "encoder.model.0" else cfg.n_filters
    g = torch.Generator().manual_seed(T * 7 + cin)
    B = 3
    x_btc = torch.randn(B, T, cin, generator=g)
    y, stats, row_off = model.debug_conv(layer, x_btc, elu=elu)
    x = x_btc.permute(0, 2, 1)
    ref = _truth(F.elu(x.double()) if elu else x, sd[layer + ".conv.conv.weight"], sd[layer + ".conv.conv.bias"])
    ref_btc = ref.permute(0, 2, 1)
    y = y.cpu().double()
    assert row_off == 0 and y.shape == ref_btc.shape, (y.shape, ref_btc.shape)
    rms = ref_btc.pow(2).mean().sqrt().item()
    err = (y - ref_btc).abs().max().item()
    print(f"{layer} T={T} C_out={ref.shape[1]} max-abs err {err:.3e} rel {err / rms:.3e}")
    assert err <= 2e-5 * rms
    st = stats.cpu().double()
    mean, var = ref.mean(dim=(1, 2)), ref.var(dim=(1, 2), unbiased=False)     # GroupNorm(1, C): over C x T
    assert (st[:, 0] - mean).abs().max().item() <= 1e-5 * rms
    assert ((st[:, 1] - 1.0 / torch.sqrt(var + 1e-5)) * torch.sqrt(var + 1e-5)).abs().max().item() <= 1e-5


# ------------------------------------------------------------------------------------------------ full width
@PATHS
def test_stereo_full_width_vs_oracle(use_tc):
    cfg, sd, model, oracle = _model("encodec_48k_stereo", 0, use_tc)
    g = torch.Generator().manual_seed(48)
    L = 3 * cfg.sample_rate
    wav = 0.1 * torch.randn(2, 2, L, generator=g)
    wav[1, 1] = 0.3 * wav[1, 0] + 0.02 * torch.randn(L, generator=g)
    ora = oracle.inference(wav, want_margin=True)
    r = model.inference(wav, need_recon=True)
    res = assert_codes_parity(_np(r["code_indices"][0]), _np(ora["code_indices"][0]), _np(ora["margins"]), MARGIN_E2E,
                              what=f"encodec_48k_stereo 2x3s {'tc' if use_tc else 'simt'}")
    scale = _np(r["code_embeddings"][0][1])
    assert np.abs(scale - _np(ora["code_embeddings"][0][1])).max() <= 1e-6 * np.abs(scale).max()
    recon = _np(r["recon_speech"])
    assert recon.shape == (2, 2, L)
    ok_clip = ~(res["first_stage"] >= 0).any(axis=1)
    for b in np.nonzero(ok_clip)[0]:
        assert np.abs(recon[b] - _np(ora["recon_speech"][b])).max() <= WAV_TOL
    d = model.inference_decoding_emb(ora["code_embeddings"][0][0])
    dref = oracle.inference_decoding_emb(ora["code_embeddings"][0][0])["recon_speech"]
    assert np.abs(_np(d["recon_speech"]) - _np(dref)).max() <= WAV_TOL


# ------------------------------------------------------------------------------------------------ properties
@PATHS
def test_stereo_properties(use_tc):
    cfg, sd, model, _ = _model("stereo_small", 0, use_tc)
    g = torch.Generator().manual_seed(5)
    L = 40 * 37 + 11
    wav = 0.1 * torch.randn(16, 2, L, generator=g)
    wav[:, 1] *= torch.linspace(0.2, 2.0, 16).view(16, 1)
    r1 = model.inference(wav, need_recon=True)
    r2 = model.inference(wav, need_recon=True)
    # determinism
    assert torch.equal(r1["code_indices"][0], r2["code_indices"][0])
    assert torch.equal(r1["recon_speech"], r2["recon_speech"])
    # batch independence: clip 5 alone == clip 5 inside B = 16 (codes and scale exactly; the waveform up to the last bits, as
    # for mono: the conv grid, and so the order in which GroupNorm partials are summed, follows the batch size)
    one = model.inference(wav[5:6], need_recon=True)
    assert torch.equal(one["code_indices"][0][:, 0], r1["code_indices"][0][:, 5])
    assert torch.equal(one["code_embeddings"][0][1][0], r1["code_embeddings"][0][1][5])
    assert (one["recon_speech"][0] - r1["recon_speech"][5]).abs().max().item() <= 1e-6
    # scale = 1e-8 + sqrt(mean(((L + R) / 2)^2)), one value per clip
    mono = (wav[:, 0] + wav[:, 1]) * 0.5
    want = 1e-8 + mono.pow(2).mean(dim=-1).sqrt()
    got = r1["code_embeddings"][0][1].view(-1).cpu()
    assert (got - want).abs().max().item() <= 1e-6 * want.abs().max().item()
    # both channels equal to one mono signal: the mono scale of that signal
    m = wav[:, 0]
    same = model.inference(torch.stack([m, m], dim=1), need_recon=False)
    mono_scale = 1e-8 + m.pow(2).mean(dim=-1).sqrt()
    assert (same["code_embeddings"][0][1].view(-1).cpu() - mono_scale).abs().max().item() <= 1e-6 * mono_scale.max().item()


def test_stereo_refusals():
    from funcodec_b200.encodec import B200Encodec
    _, _, stereo, _ = _model("stereo_small", 0, 1)
    _, _, mono, _ = _model("tiny_ds40", 0, 1)
    with pytest.raises(ValueError, match="only mono"):
        mono.inference(torch.zeros(1, 2, 400))
    for bad in (torch.zeros(1, 400), torch.zeros(1, 1, 400), torch.zeros(1, 3, 400)):
        with pytest.raises(ValueError, match="stereo"):
            stereo.inference(bad)
    import dataclasses
    cfg = dataclasses.replace(get_config("freq_small"), channels=2)
    with pytest.raises(FcbError, match="fcb_create"):
        B200Encodec(cfg, {}, "cuda:0")
