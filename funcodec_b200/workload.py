"""Analytic work model of the hot path (host logic): multiply-accumulates, layer-boundary bytes and parameter counts of the
SEANet stacks, the SLSTMs and the RVQ for a CodecConfig and an input length.

It restates SURVEY.md §8(d)'s accounting -- which was probed on the reference modules with forward hooks -- so that the roofline
numerators bench.py quotes (its per-config constants) can be re-derived and are checked on CPU (tests/test_workload.py), and it
is what `--stat_flops` logs in place of the reference's thop profile (codec_inference.py:329-345):

  * conv MACs: T_out * C_in / groups * C_out * k per conv (x F_out, x k_f in 2-D); a transposed conv does T_in * C_in * C_out * k
  * layer-boundary bytes: 4 * (|module input| + |module output|) per conv / transposed-conv MODULE as the hooks see them: the
    conv input is the padded tensor (SConv pads before calling the conv), the transposed-conv output is the untrimmed one
  * LSTM MACs: 2 stacks x layers x T' x 8 H^2 (W_ih and W_hh, 4 gates);  RVQ FLOPs: 2 * T' * n_q * K * D
  * stereo (cfg.channels = 2): the first conv reads and the last conv writes 2 channels per sample; L counts samples per channel
"""
from typing import Dict

from .config import CodecConfig


def _time_stacks(cfg: CodecConfig, L: int, layers=None):
    nf, D = cfg.n_filters, cfg.dimension
    macs = byts = params = 0
    nres = cfg.n_residual_layers

    def note(name, cin, cout, k, s, To, m, b):
        if layers is not None:
            layers.append(dict(name=name, cin=cin, cout=cout, k=k, s=s, T_out=To, macs=m, bytes=b))

    def conv(cin, cout, k, s, T, d=1, name="conv"):
        nonlocal macs, byts, params
        To = -(-T // s)
        Tp = (To - 1) * s + (k - 1) * d + 1                 # padded input length (reflect padding incl. the extra padding)
        macs += To * cin * cout * k
        byts += 4 * (Tp * cin + To * cout)
        note(name, cin, cout, k, s, To, To * cin * cout * k, 4 * (Tp * cin + To * cout))
        params += cin * cout * k + cout + (2 * cout if cfg.norm == "time_group_norm" else (cout if cfg.norm == "weight_norm" else 0))
        return To

    def lstm_inputs(side, T, H):
        # the W_ih half of each LSTM layer runs as a 1x1 GEMM launch of the conv kernel (its MACs belong to lstm_macs)
        for l in range(cfg.lstm_layers):
            note(f"{side}.lstm.ih_l{l}", H, 4 * H, 1, 1, T, T * H * 4 * H, 4 * (T * H + T * 4 * H))

    T = conv(cfg.channels, nf, cfg.kernel_size, 1, L, name="enc.conv0")
    mult = 1
    for i, r in enumerate(reversed(cfg.ratios)):
        for j in range(nres):
            conv(mult * nf, mult * nf // 2, cfg.residual_kernel_size, 1, T, cfg.dilation_base ** j, name=f"enc.{i}.rb{j}.k3")
            conv(mult * nf // 2, mult * nf, 1, 1, T, name=f"enc.{i}.rb{j}.1x1")
            conv(mult * nf, mult * nf, 1, 1, T, name=f"enc.{i}.rb{j}.shortcut")
        T = conv(mult * nf, 2 * mult * nf, 2 * r, r, T, name=f"enc.{i}.down")
        mult *= 2
    H = mult * nf
    lstm_inputs("enc", T, H)
    conv(H, D, cfg.last_kernel_size, 1, T, name="enc.final")
    frames = T
    conv(D, H, cfg.kernel_size, 1, T, name="dec.conv0")
    lstm_inputs("dec", T, H)
    for i, r in enumerate(cfg.ratios):
        cin, cout, k = mult * nf, mult * nf // 2, 2 * r
        macs += T * cin * cout * k
        byts += 4 * (T * cin + (T + 1) * r * cout)           # ConvTranspose1d output before unpad1d: (T - 1) r + 2 r
        note(f"dec.{i}.up", cin, cout, k, r, T * r, T * cin * cout * k, 4 * (T * cin + (T + 1) * r * cout))
        params += cin * cout * k + cout + (2 * cout if cfg.norm == "time_group_norm" else (cin if cfg.norm == "weight_norm" else 0))
        T *= r
        for j in range(nres):
            conv(cout, cout // 2, cfg.residual_kernel_size, 1, T, cfg.dilation_base ** j, name=f"dec.{i}.rb{j}.k3")
            conv(cout // 2, cout, 1, 1, T, name=f"dec.{i}.rb{j}.1x1")
            conv(cout, cout, 1, 1, T, name=f"dec.{i}.rb{j}.shortcut")
        mult //= 2
    conv(nf, cfg.channels, cfg.last_kernel_size, 1, T, name="dec.final")
    return macs, byts, params, frames, H


def _freq_stacks(cfg: CodecConfig, L: int):
    nf, D, rk = cfg.n_filters, cfg.dimension, cfg.residual_kernel_size
    F, T = cfg.n_fft // 2 + 1, 1 + L // cfg.stft_hop
    macs = byts = params = 0

    def conv2(cin, cout, kf, kt, sf, st, F, T, groups=1):
        nonlocal macs, byts, params
        Fo, To = (F - sf) // sf + 1, -(-T // st)             # frequency: fixed padding k - s, no extra; time: like SConv1d
        Fp, Tp = F + kf - sf, (To - 1) * st + kt
        macs += Fo * To * (cin // groups) * cout * kf * kt
        byts += 4 * (Fp * Tp * cin + Fo * To * cout)
        params += (cin // groups) * cout * kf * kt + 3 * cout
        return Fo, To

    def resblock(dim, F, T):
        g = cfg.conv_groups(dim // 2)
        conv2(dim, dim // 2, rk, rk, 1, 1, F, T, g)
        conv2(dim // 2, dim, 1, 1, 1, 1, F, T, g)
        conv2(dim, dim, 1, 1, 1, 1, F, T, cfg.conv_groups(dim))

    conv2(3, nf, cfg.kernel_size, cfg.kernel_size, 1, 1, F, T)
    mult = 1
    for fr, tr in reversed(list(zip(cfg.ratios_f, cfg.ratios))):
        resblock(mult * nf, F, T)
        F, T = conv2(mult * nf, 2 * mult * nf, 2 * fr, 2 * tr, fr, tr, F, T, cfg.conv_groups(mult * nf))
        mult *= 2
    if F != 1:
        raise ValueError(f"the frequency ratios leave {F} bins, not 1")
    H, frames = mult * nf, T
    for cin, cout, k in ((H, D, cfg.last_kernel_size), (D, H, cfg.kernel_size)):      # the two 1-D convs around the RVQ
        macs += T * cin * cout * k
        byts += 4 * ((T + k - 1) * cin + T * cout)
        params += cin * cout * k + 3 * cout
    n_st = len(cfg.ratios)
    for i, (fr, tr) in enumerate(zip(cfg.ratios_f, cfg.ratios)):
        cin, cout, g = mult * nf, mult * nf // 2, cfg.tr_conv_groups(mult * nf)
        macs += F * T * cin * (cout // g) * 2 * fr * 2 * tr
        byts += 4 * (F * T * cin + (F + 1) * fr * (T + 1) * tr * cout)                  # untrimmed ConvTranspose2d output
        params += cin * (cout // g) * 4 * fr * tr + 3 * cout
        F, T = F * fr + (1 if i == n_st - 1 else 0), T * tr                             # last stage: out_padding restores n_fft/2 + 1
        resblock(cout, F, T)
        mult //= 2
    conv2(nf, 3, cfg.last_kernel_size, cfg.last_kernel_size, 1, 1, F, T)
    return macs, byts, params, frames, H


def conv_launches(cfg: CodecConfig, L: int):
    """The conv-kernel launches of one time-domain round trip in the engine's launch order (per clip): name, shape, MACs and
    layer-boundary bytes of each -- what tools/per_layer_roofline.py lines up with an ncu launch list."""
    if cfg.arch != 0:
        raise ValueError("per-launch list: time-domain stacks only")
    layers = []
    _time_stacks(cfg, L, layers)
    return layers


def workload_model(cfg: CodecConfig, L: int, n_q: int = 0) -> Dict[str, float]:
    """Per CLIP of L samples.  Keys: conv_macs, conv_bytes (layer-boundary model, fp32), lstm_macs, rvq_flops, frames,
    conv_params / lstm_params / codebook_params (scalars; x 4 = bytes), weight_bytes (conv + LSTM, what SURVEY adds once per
    batch), total_macs (conv + LSTM + RVQ as MACs)."""
    n_q = n_q or cfg.num_quantizers
    macs, byts, params, frames, H = (_freq_stacks if cfg.arch == 1 else _time_stacks)(cfg, L)
    lstm_macs = 2 * cfg.lstm_layers * frames * 8 * H * H
    lstm_params = 2 * cfg.lstm_layers * (8 * H * H + 8 * H)
    rvq_flops = 2 * frames * n_q * cfg.codebook_size * cfg.dimension
    return dict(conv_macs=float(macs), conv_bytes=float(byts), lstm_macs=float(lstm_macs), rvq_flops=float(rvq_flops),
                frames=int(frames), conv_params=int(params), lstm_params=int(lstm_params),
                codebook_params=int(cfg.num_quantizers * cfg.codebook_size * cfg.dimension),
                weight_bytes=float(4 * (params + lstm_params)),       # every parameter tensor of the stacks, as SURVEY counts them
                total_macs=float(macs + lstm_macs + rvq_flops / 2))

