"""Parameter naming (the reference's state_dict keys, SURVEY.md App. D) and a seeded synthetic init.

There is no network for pretrained checkpoints, so bench/tests use `init_state_dict(cfg, seed)`:
reference-shaped tensors under the reference's names, drawn with a seeded CPU generator so that
the CUDA path, the oracle and (in the build container) the real reference modules all consume
bit-identical weights.  Host logic only.
"""
from typing import Dict, List, Tuple
import math
import torch

from .config import CodecConfig


def conv_specs(cfg: CodecConfig) -> List[Dict]:
    """Every conv / transposed conv of encoder+decoder in execution order, with reference names.
    Encoder: funcodec/models/encoder/seanet_encoder.py:108-162; decoder: seanet_decoder.py:107-172."""
    specs = []
    nf, D = cfg.n_filters, cfg.dimension

    def rb(prefix, dim):
        return [dict(name=prefix + ".block.1.conv", kind="conv", cin=dim, cout=dim // 2, k=cfg.residual_kernel_size, s=1),
                dict(name=prefix + ".block.3.conv", kind="conv", cin=dim // 2, cout=dim, k=1, s=1),
                dict(name=prefix + ".shortcut.conv", kind="conv", cin=dim, cout=dim, k=1, s=1)]

    specs.append(dict(name="encoder.model.0.conv", kind="conv", cin=cfg.channels, cout=nf, k=cfg.kernel_size, s=1))
    n, mult = 1, 1
    nres = cfg.n_residual_layers
    for r in reversed(cfg.ratios):
        for j in range(nres):
            specs += rb(f"encoder.model.{n + j}", mult * nf)
        specs.append(dict(name=f"encoder.model.{n + nres + 1}.conv", kind="conv", cin=mult * nf, cout=2 * mult * nf, k=2 * r, s=r))
        mult *= 2
        n += nres + 2
    if cfg.lstm_layers > 0:
        specs.append(dict(name=f"encoder.model.{n}.lstm", kind="lstm", dim=mult * nf))
        n += 1
    specs.append(dict(name=f"encoder.model.{n + 1}.conv", kind="conv", cin=mult * nf, cout=D, k=cfg.last_kernel_size, s=1))

    specs.append(dict(name="decoder.model.0.conv", kind="conv", cin=D, cout=mult * nf, k=cfg.kernel_size, s=1))
    n = 1
    if cfg.lstm_layers > 0:
        specs.append(dict(name="decoder.model.1.lstm", kind="lstm", dim=mult * nf))
        n = 2
    for r in cfg.ratios:
        specs.append(dict(name=f"decoder.model.{n + 1}.convtr", kind="convtr", cin=mult * nf, cout=mult * nf // 2, k=2 * r, s=r))
        for j in range(nres):
            specs += rb(f"decoder.model.{n + 2 + j}", mult * nf // 2)
        mult //= 2
        n += nres + 2
    specs.append(dict(name=f"decoder.model.{n + 1}.conv", kind="conv", cin=nf, cout=cfg.channels, k=cfg.last_kernel_size, s=1))
    return specs


def _freq_shapes(cfg: CodecConfig) -> Dict[str, Tuple[int, ...]]:
    """SEANetEncoder2d / SEANetDecoder2d parameter names and shapes (seanet_encoder.py:252-363, seanet_decoder.py:244-360),
    grouped like the reference when cfg.conv_group_ratio / tr_conv_group_ratio > 0."""
    sh: Dict[str, Tuple[int, ...]] = {}
    nf, D, rk = cfg.n_filters, cfg.dimension, cfg.residual_kernel_size

    def conv2(name, cin, cout, kf, kt, groups=1):
        sh[name + ".conv.conv.weight"] = (cout, cin // groups, kf, kt); sh[name + ".conv.conv.bias"] = (cout,)
        sh[name + ".conv.norm.weight"] = (cout,); sh[name + ".conv.norm.bias"] = (cout,)

    def conv1(name, cin, cout, k):
        sh[name + ".conv.conv.weight"] = (cout, cin, k); sh[name + ".conv.conv.bias"] = (cout,)
        sh[name + ".conv.norm.weight"] = (cout,); sh[name + ".conv.norm.bias"] = (cout,)

    def rb(name, dim):
        g = cfg.conv_groups(dim // 2)                    # min(in, out) = dim // 2 for both block convs
        conv2(name + ".block.1", dim, dim // 2, rk, rk, g); conv2(name + ".block.3", dim // 2, dim, 1, 1, g)
        conv2(name + ".shortcut", dim, dim, 1, 1, cfg.conv_groups(dim))

    def lstm(name, H):
        for l in range(cfg.lstm_layers):
            sh[f"{name}.lstm.weight_ih_l{l}"] = (4 * H, H); sh[f"{name}.lstm.weight_hh_l{l}"] = (4 * H, H)
            sh[f"{name}.lstm.bias_ih_l{l}"] = (4 * H,); sh[f"{name}.lstm.bias_hh_l{l}"] = (4 * H,)

    conv2("encoder.model.0", 3, nf, cfg.kernel_size, cfg.kernel_size)
    n, mult = 1, 1
    for fr, tr in reversed(list(zip(cfg.ratios_f, cfg.ratios))):
        rb(f"encoder.model.{n}", mult * nf)
        conv2(f"encoder.model.{n + 2}", mult * nf, 2 * mult * nf, 2 * fr, 2 * tr, cfg.conv_groups(mult * nf))
        mult *= 2; n += 3
    n += 1
    if cfg.lstm_layers > 0:
        lstm(f"encoder.model.{n}", mult * nf); n += 1
    conv1(f"encoder.model.{n + 1}", mult * nf, D, cfg.last_kernel_size)
    conv1("decoder.model.0", D, mult * nf, cfg.kernel_size)
    n = 1
    if cfg.lstm_layers > 0:
        lstm("decoder.model.1", mult * nf); n = 2
    n += 1
    for fr, tr in zip(cfg.ratios_f, cfg.ratios):
        name = f"decoder.model.{n + 1}"
        sh[name + ".convtr.convtr.weight"] = (mult * nf, mult * nf // 2 // cfg.tr_conv_groups(mult * nf), 2 * fr, 2 * tr)
        sh[name + ".convtr.convtr.bias"] = (mult * nf // 2,)
        sh[name + ".convtr.norm.weight"] = (mult * nf // 2,); sh[name + ".convtr.norm.bias"] = (mult * nf // 2,)
        rb(f"decoder.model.{n + 2}", mult * nf // 2)
        mult //= 2; n += 3
    conv2(f"decoder.model.{n + 1}", nf, 3, cfg.last_kernel_size, cfg.last_kernel_size)
    nq, K = cfg.num_quantizers, cfg.codebook_size
    sh["quantizer.rq.model.inited"] = (nq, 1); sh["quantizer.rq.model.cluster_size"] = (nq, K)
    sh["quantizer.rq.model.embed"] = (nq, K, D); sh["quantizer.rq.model.embed_avg"] = (nq, K, D)
    return sh


def state_dict_shapes(cfg: CodecConfig) -> Dict[str, Tuple[int, ...]]:
    if cfg.arch == 1:
        return _freq_shapes(cfg)
    shapes: Dict[str, Tuple[int, ...]] = {}
    def normed(base, wshape, cout):
        # NormConv1d / NormConvTranspose1d parameters (conv.py:25-55,148-202): weight_norm re-parametrises `weight` as
        # weight_g [d0,1,1] x weight_v and has no norm module; 'none' has neither
        if cfg.norm == "weight_norm":
            shapes[base + ".weight_v"] = wshape
            shapes[base + ".weight_g"] = (wshape[0], 1, 1)
        else:
            shapes[base + ".weight"] = wshape
        shapes[base + ".bias"] = (cout,)
        if cfg.norm == "time_group_norm":
            head = base.rsplit(".", 1)[0]
            shapes[head + ".norm.weight"] = (cout,)
            shapes[head + ".norm.bias"] = (cout,)

    for sp in conv_specs(cfg):
        n = sp["name"]
        if sp["kind"] == "conv":
            normed(n + ".conv", (sp["cout"], sp["cin"], sp["k"]), sp["cout"])
        elif sp["kind"] == "convtr":
            normed(n + ".convtr", (sp["cin"], sp["cout"], sp["k"]), sp["cout"])
        else:
            H = sp["dim"]
            for l in range(cfg.lstm_layers):
                shapes[f"{n}.weight_ih_l{l}"] = (4 * H, H)
                shapes[f"{n}.weight_hh_l{l}"] = (4 * H, H)
                shapes[f"{n}.bias_ih_l{l}"] = (4 * H,)
                shapes[f"{n}.bias_hh_l{l}"] = (4 * H,)
    nq, K, D = cfg.num_quantizers, cfg.codebook_size, cfg.dimension
    # use_ddp=True buffers (funcodec/modules/quantization/ddp_core_vq.py:349-352)
    shapes["quantizer.rq.model.inited"] = (nq, 1)
    shapes["quantizer.rq.model.cluster_size"] = (nq, K)
    shapes["quantizer.rq.model.embed"] = (nq, K, D)
    shapes["quantizer.rq.model.embed_avg"] = (nq, K, D)
    return shapes


WN_GAIN = 1.6


def init_state_dict(cfg: CodecConfig, seed: int = 0) -> Dict[str, torch.Tensor]:
    """Seeded synthetic weights: conv/LSTM ~ U(-1/sqrt(fan_in), 1/sqrt(fan_in)) like torch's defaults,
    GroupNorm affine perturbed away from (1, 0) so the affine path is exercised, codebooks
    N(0, sigma_q^2) with geometrically shrinking sigma_q (residuals shrink stage by stage)."""
    g = torch.Generator().manual_seed(seed)
    sd: Dict[str, torch.Tensor] = {}

    def uni(shape, bound):
        return (torch.rand(shape, generator=g, dtype=torch.float32) * 2 - 1) * bound

    for name, shape in state_dict_shapes(cfg).items():
        if name.startswith("quantizer."):
            continue
        if name.endswith("norm.weight"):
            sd[name] = 1.0 + 0.1 * torch.randn(shape, generator=g)
        elif name.endswith("norm.bias"):
            sd[name] = 0.1 * torch.randn(shape, generator=g)
        elif ".lstm." in name:
            H = shape[-1] if len(shape) == 2 else shape[0] // 4
            sd[name] = uni(shape, 1.0 / math.sqrt(H))
        elif name.endswith("convtr.weight") or name.endswith("conv.weight") or name.endswith(".weight_v"):
            fan_in = shape[1] * int(math.prod(shape[2:]))     # torch: fan_in uses dim 1 (also for [Cin, Cout, k...])
            sd[name] = uni(shape, 1.0 / math.sqrt(fan_in))
        elif name.endswith(".weight_g"):
            # weight_norm initialises g = ||v|| (so w == v); perturbed, and with the gain that keeps activations O(1) through the
            # un-normalised stack (v ~ U(+-1/sqrt(fan_in)) alone shrinks the variance 3x per conv)
            v = sd[name[:-1] + "v"]
            sd[name] = v.flatten(1).norm(dim=1).view(shape) * WN_GAIN * (1.0 + 0.1 * torch.randn(shape, generator=g))
        else:  # conv / convtr bias
            sd[name] = uni(shape, 0.1)
    nq, K, D = cfg.num_quantizers, cfg.codebook_size, cfg.dimension
    sigma = 0.6 * (0.93 ** torch.arange(nq, dtype=torch.float32)).view(nq, 1, 1)
    embed = torch.randn((nq, K, D), generator=g) * sigma
    sd["quantizer.rq.model.inited"] = torch.ones(nq, 1)
    sd["quantizer.rq.model.cluster_size"] = torch.ones(nq, K)
    sd["quantizer.rq.model.embed"] = embed
    sd["quantizer.rq.model.embed_avg"] = embed.clone()
    return sd
