"""Pin the CPU oracle (oracle/encodec_oracle.py) against vectors produced by the UNMODIFIED
reference modules (tools/gen_golden.py -> tests/golden/*.npz).  CPU only.

ATen CPU kernels are deterministic for a fixed thread count but conv/GEMM blocking can differ
between hosts, so the pin is 'equal codes + 2e-6 max-abs' rather than bitwise equality.
"""
import os

import numpy as np
import pytest
import torch

from funcodec_b200 import get_config, init_state_dict
from oracle import encodec_oracle as O

TOL = 2e-6
# the vectors were generated with 8 intra-op threads; with fewer, ATen splits some float32 reductions differently and the
# deeper model outputs move by a few 1e-6 (3 threads: up to 5e-6), so the oracle runs with the same count
GOLDEN_THREADS = 8


@pytest.fixture(autouse=True, scope="module")
def _golden_threads():
    n = torch.get_num_threads()
    torch.set_num_threads(GOLDEN_THREADS)
    yield
    torch.set_num_threads(n)


def _load(golden_dir, name):
    return np.load(os.path.join(golden_dir, name))


def _sd_checksum(sd):
    return float(sum(v.double().abs().sum().item() for v in sd.values()))


def test_layers_conv(golden_dir):
    z = _load(golden_dir, "layers.npz")
    for i in range(int(z["n_conv"])):
        pre = f"conv{i}."
        cin, cout, k, s, d, T = z[pre + "meta"]
        p = {"m.conv.conv.weight": torch.from_numpy(z[pre + "w"]), "m.conv.conv.bias": torch.from_numpy(z[pre + "b"]),
             "m.conv.norm.weight": torch.from_numpy(z[pre + "gw"]), "m.conv.norm.bias": torch.from_numpy(z[pre + "gb"])}
        y = O.sconv1d(torch.from_numpy(z[pre + "x"]), p, "m", stride=int(s), dilation=int(d))
        assert y.shape == z[pre + "y"].shape
        assert np.abs(y.numpy() - z[pre + "y"]).max() <= TOL, (i, cin, cout, k, s, d, T)


def test_layers_convtr(golden_dir):
    z = _load(golden_dir, "layers.npz")
    for i in range(int(z["n_convtr"])):
        pre = f"convtr{i}."
        cin, cout, k, s, T = z[pre + "meta"]
        p = {"m.convtr.convtr.weight": torch.from_numpy(z[pre + "w"]), "m.convtr.convtr.bias": torch.from_numpy(z[pre + "b"]),
             "m.convtr.norm.weight": torch.from_numpy(z[pre + "gw"]), "m.convtr.norm.bias": torch.from_numpy(z[pre + "gb"])}
        y = O.sconvtr1d(torch.from_numpy(z[pre + "x"]), p, "m", stride=int(s))
        assert y.shape == z[pre + "y"].shape == (2, cout, T * s)
        assert np.abs(y.numpy() - z[pre + "y"]).max() <= TOL


def test_layers_resblock_lstm(golden_dir):
    z = _load(golden_dir, "layers.npz")
    p = {"m." + k[len("rb.sd."):]: torch.from_numpy(z[k]) for k in z.files if k.startswith("rb.sd.")}
    y = O.resblock(torch.from_numpy(z["rb.x"]), p, "m")
    assert np.abs(y.numpy() - z["rb.y"]).max() <= TOL
    p = {"m." + k[len("lstm.sd."):]: torch.from_numpy(z[k]) for k in z.files if k.startswith("lstm.sd.")}
    x = torch.from_numpy(z["lstm.x"])
    for manual in (False, True):   # the explicit-loop restatement must agree with nn.LSTM too
        y = O.slstm(x, p, "m", 2, manual=manual)
        assert np.abs(y.numpy() - z["lstm.y"]).max() <= TOL


def test_layers_rvq(golden_dir):
    z = _load(golden_dir, "layers.npz")
    embed = torch.from_numpy(z["rvq.embed"])
    x = torch.from_numpy(z["rvq.x"])
    quant, codes, sub, margins = O.rvq_forward(x, embed, 6, want_margin=True)
    assert np.array_equal(codes.numpy(), z["rvq.codes"])
    assert np.abs(quant.numpy() - z["rvq.quant"]).max() <= TOL
    assert np.abs(sub.numpy() - z["rvq.sub"]).max() == 0
    assert (margins >= 0).all()
    quant4, codes4, _, _ = O.rvq_forward(x, embed, 4)
    assert np.array_equal(codes4.numpy(), z["rvq.codes4"])
    assert np.abs(quant4.numpy() - z["rvq.quant4"]).max() <= TOL
    dec = O.rvq_decode(codes, embed)
    assert np.abs(dec.numpy() - z["rvq.decode"]).max() <= TOL


MODEL_FILES = ["model_tiny_ds40.npz", "model_tiny_ds40_ragged.npz", "model_small_ds320.npz",
               "model_encodec_16k_n32_ds640.npz", "model_encodec_16k_n32_ds320.npz",
               # norm weight_norm: {causal, 3 dilated residual blocks, no sequence model} and {non-causal, SLSTM}
               # (tools/gen_golden_norms.py)
               "model_soundstream_causal_small.npz", "model_weightnorm_lstm_small.npz"]


@pytest.mark.parametrize("fname", MODEL_FILES)
def test_model_inference(golden_dir, fname):
    z = _load(golden_dir, fname)
    cfg = get_config(str(z["cfg_name"]))
    sd = init_state_dict(cfg, int(z["seed"]))
    assert abs(_sd_checksum(sd) - float(z["sd_checksum"])) <= 1e-6 * float(z["sd_checksum"]), "synthetic init drifted"
    o = O.OracleEncodec.from_config(sd, cfg)
    wav = torch.from_numpy(z["wav"])
    keys = sorted({k.split(".")[0] for k in z.files if k.endswith(".codes")})
    for key in keys:
        bw = None if key == "full" else int(key[2:])
        r = o.inference(wav, need_recon=True, bit_width=bw, use_scale=True)
        assert np.array_equal(r["code_indices"][0].numpy(), z[f"{key}.codes"].astype(np.int64)), key
        assert np.abs(r["code_embeddings"][0][0].numpy() - z[f"{key}.quant"]).max() <= TOL
        assert np.abs(r["code_embeddings"][0][1].numpy() - z[f"{key}.scale"]).max() <= 1e-7
        assert r["recon_speech"].shape == z[f"{key}.recon"].shape == (wav.shape[0], 1, wav.shape[1])
        assert np.abs(r["recon_speech"].numpy() - z[f"{key}.recon"]).max() <= TOL
    r = o.inference(wav)
    assert np.abs(r["encoder_out"].numpy() - z["encoder_out"]).max() <= TOL
    assert np.allclose(r["sub_quants"][0].double().sum(dim=(2, 3)).numpy(), z["full.sub_quants_sum"], atol=1e-4)
    toks = r["code_indices"][0].permute(1, 2, 0)
    d = o.inference_decoding(toks)
    assert np.abs(d["recon_speech"].numpy() - z["decode_codes.recon"]).max() <= TOL
    d = o.inference_decoding_emb(r["code_embeddings"][0][0])
    assert np.abs(d["recon_speech"].numpy() - z["decode_emb.recon"]).max() <= TOL
    r2 = o.inference(wav, use_scale=False)
    assert np.abs(r2["recon_speech"].numpy() - z["noscale.recon"]).max() <= TOL


def test_padding_arithmetic_property():
    """SURVEY App. B: T_out == ceil(T / s) for every (k, s) family; reflect pad never reads OOB."""
    for (k, s) in [(7, 1), (3, 1), (1, 1), (4, 2), (8, 4), (10, 5), (16, 8)]:
        for T in list(range(1, 70)) + [160000, 479999]:
            pl, pr = O.conv_paddings(T, k, s, 1)
            t_out = (T + pl + pr - k) // s + 1
            assert t_out == -(-T // s), (k, s, T)
            assert (T + pl + pr - k) % s == 0


def test_numpy_cross_check_conv_groupnorm():
    """Independent numpy restatement (explicit loops) of reflect-pad conv + GroupNorm(1,C) on a small case,
    so the torch-functional oracle is not the only statement of the algorithm."""
    rng = np.random.default_rng(0)
    cin, cout, k, s, T = 3, 4, 4, 2, 11
    x = rng.standard_normal((1, cin, T)).astype(np.float32)
    w = rng.standard_normal((cout, cin, k)).astype(np.float32)
    b = rng.standard_normal(cout).astype(np.float32)
    gw = rng.standard_normal(cout).astype(np.float32)
    gb = rng.standard_normal(cout).astype(np.float32)
    pl, pr = O.conv_paddings(T, k, s, 1)

    def refl(i):
        if i < 0:
            return -i
        if i >= T:
            return 2 * (T - 1) - i
        return i
    t_out = -(-T // s)
    y = np.zeros((cout, t_out), np.float64)
    for co in range(cout):
        for t in range(t_out):
            acc = float(b[co])
            for ci in range(cin):
                for kk in range(k):
                    acc += float(w[co, ci, kk]) * float(x[0, ci, refl(t * s + kk - pl)])
            y[co, t] = acc
    mean, var = y.mean(), y.var()
    yn = (y - mean) / np.sqrt(var + 1e-5) * gw[:, None] + gb[:, None]
    p = {"m.conv.conv.weight": torch.from_numpy(w), "m.conv.conv.bias": torch.from_numpy(b),
         "m.conv.norm.weight": torch.from_numpy(gw), "m.conv.norm.bias": torch.from_numpy(gb)}
    got = O.sconv1d(torch.from_numpy(x), p, "m", stride=s).numpy()[0]
    assert np.abs(got - yn).max() < 1e-5


@pytest.mark.parametrize("tag", ["a", "b"])
def test_model_inference_segmented(golden_dir, tag):
    """segment_dur != None (codec_basic.py:287-298,334-359,382-396): per-segment scale / codes / embeddings and the
    linear overlap-add, against the unmodified reference (tools/gen_golden_seg.py)."""
    z = np.load(os.path.join(golden_dir, "model_small_ds320_segmented.npz"))
    cfg = get_config(str(z["cfg_name"]))
    sd = init_state_dict(cfg, int(z["seed"]))
    dur, ov, B, L, _, seg, stride, n_seg = z[f"{tag}.meta"]
    ora = O.OracleEncodec(sd, cfg.ratios, cfg.sample_rate, cfg.lstm_layers, segment_dur=float(dur), overlap_ratio=float(ov))
    assert O.segment_plan(int(L), cfg.sample_rate, float(dur), float(ov))[:2] == (int(seg), int(stride))
    r = ora.inference(torch.from_numpy(z[f"{tag}.wav"]))
    assert len(r["code_indices"]) == int(n_seg)
    for i in range(int(n_seg)):
        assert np.array_equal(r["code_indices"][i].numpy(), z[f"{tag}.codes{i}"].astype(np.int64))
        assert np.abs(r["code_embeddings"][i][0].numpy() - z[f"{tag}.quant{i}"]).max() <= 1e-6
        assert np.array_equal(r["code_embeddings"][i][1].numpy(), z[f"{tag}.scale{i}"])
        assert np.abs(r["encoder_out"][i].numpy() - z[f"{tag}.encoder_out{i}"]).max() <= 1e-6
    assert r["recon_speech"].shape == z[f"{tag}.recon"].shape
    assert np.abs(r["recon_speech"].numpy() - z[f"{tag}.recon"]).max() <= 1e-6


def test_overlap_add_overrun_is_an_error():
    """The reference cannot overlap-add a non-final frame that ends after the final one (codec_basic.py:112 raises);
    the oracle keeps that behaviour."""
    frames = [torch.ones(1, 1, 1920), torch.ones(1, 1, 1920), torch.ones(1, 1, 1600), torch.ones(1, 1, 640)]
    with pytest.raises(RuntimeError):
        O.linear_overlap_add(frames, 880)


def test_laura_call_patterns_on_the_oracle():
    """SURVEY §8(f) N3: the LauraTTS call patterns (tests/laura_calls.py) run against the oracle stand-in; the GPU suite
    replays the same calls through funcodec_b200.Speech2Token and compares."""
    from laura_calls import OracleSpeech2Token, laura_codec_calls
    cfg = get_config("small_ds320")
    sd = init_state_dict(cfg, 3)
    ora = O.OracleEncodec(sd, cfg.ratios, cfg.sample_rate, cfg.lstm_layers)
    g = torch.Generator().manual_seed(5)
    prompt = 0.1 * torch.randn(1, 320 * 12 + 100, generator=g)
    r = laura_codec_calls(OracleSpeech2Token(ora), prompt, sd["quantizer.rq.model.embed"])
    assert tuple(r["codec"].shape) == (13, cfg.num_quantizers) and len(r["continual"]) == 13 and len(r["continual"][0]) == 2
    assert tuple(r["gen_only_lm"].shape) == (1, 1, 13 * 320) == tuple(r["gen"].shape)
    # with exactly the predicted groups, decoding the codes and decoding their summed codewords are the same computation
    assert (r["gen_only_lm"] - r["gen"]).abs().max().item() <= 1e-5


def test_soundstream_noncausal_topology(golden_dir):
    """conf/soundstream_noncausal_16k_n32_600k_step.yaml's topology -- three residual blocks per stage with dilations 1 / 2 / 4
    (seanet_encoder.py:122-128), no sequence model -- against the unmodified reference SEANetEncoder / SEANetDecoder
    (tools/gen_golden_soundstream.py).  (The CUDA engine builds this topology too: tests/test_gpu_parity.py.)"""
    z = np.load(os.path.join(golden_dir, "soundstream_noncausal_small.npz"))
    sd = {k[3:]: torch.from_numpy(z[k]) for k in z.files if k.startswith("sd.")}
    ratios = [int(r) for r in z["ratios"]]
    emb = O.seanet_encoder(torch.from_numpy(z["x"]), O.sub_dict(sd, "encoder."), ratios, lstm_layers=0, n_residual_layers=3)
    assert emb.shape == z["emb"].shape
    assert np.abs(emb.numpy() - z["emb"]).max() <= 2e-6
    y = O.seanet_decoder(torch.from_numpy(z["emb"]), O.sub_dict(sd, "decoder."), ratios, lstm_layers=0, n_residual_layers=3)
    assert y.shape == z["y"].shape
    assert np.abs(y.numpy() - z["y"]).max() <= 2e-6


def test_soundstream_causal_weight_norm_topology(golden_dir):
    """conf/soundstream_16k_n32_600k_step.yaml's branches -- `norm: weight_norm` (weight_g / weight_v re-parametrisation, no norm
    module, conv.py:25-55) and `causal: true` (left-only reflect padding, right-only trimming of the transposed convs,
    conv.py:251-253,293-297) on the stacked dilated residual blocks -- against the unmodified reference SEANetEncoder /
    SEANetDecoder (tools/gen_golden_soundstream.py)."""
    z = np.load(os.path.join(golden_dir, "soundstream_causal_small.npz"))
    sd = {k[3:]: torch.from_numpy(z[k]) for k in z.files if k.startswith("sd.")}
    assert "encoder.model.0.conv.conv.weight_g" in sd and "encoder.model.0.conv.norm.weight" not in sd
    ratios = [int(r) for r in z["ratios"]]
    kw = dict(lstm_layers=0, n_residual_layers=3, causal=True)
    emb = O.seanet_encoder(torch.from_numpy(z["x"]), O.sub_dict(sd, "encoder."), ratios, **kw)
    assert emb.shape == z["emb"].shape
    assert np.abs(emb.numpy() - z["emb"]).max() <= 2e-6
    y = O.seanet_decoder(torch.from_numpy(z["emb"]), O.sub_dict(sd, "decoder."), ratios, **kw)
    assert y.shape == z["y"].shape
    assert np.abs(y.numpy() - z["y"]).max() <= 2e-6
    # the non-causal paddings on the same weights give a different signal (the flag is live)
    emb_nc = O.seanet_encoder(torch.from_numpy(z["x"]), O.sub_dict(sd, "encoder."), ratios, lstm_layers=0, n_residual_layers=3)
    assert np.abs(emb_nc.numpy() - z["emb"]).max() > 1e-3
