"""Throughput of the stereo time-domain Encodec (preset encodec_48k_stereo) on one GPU, next to the mono
encodec_16k_n32_ds640 step at the same batch.  Prints one JSON line.

Legs (B clips of S seconds each, one fcb_roundtrip per step: normalise, encode, RVQ at full n_q, decode):
  stereo_whole      encodec_48k_stereo, whole clips [B, 2, S * 48000]
  stereo_segmented  the same clips with segment_dur 1.0 / overlap_ratio 0.01 (Encodec's defaults, codec_basic.py:143-144):
                    fcb_roundtrip_segmented, per-segment scale, overlap-add
  mono_ds640        encodec_16k_n32_ds640 on [B, S * 16000] (the workload of bench.py's config 2 at this batch)

Method: every leg warms up on the timed shapes, rotates its inputs over enough distinct batches (> 140 MB) that no step reads
an L2-resident input (126 MB L2), and times `--steps` back-to-back steps between two CUDA events.  The per-phase split is
fcb_get_phase_ms of the last timed step (whole-clip legs).  The card's name and power limit are read in the same run.
Run:  python tools/bench_stereo.py [--batch 16] [--seconds 10] [--steps 10] [--warmup 3]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from funcodec_b200 import get_config, init_state_dict  # noqa: E402
from funcodec_b200.encodec import B200Encodec, _ptr  # noqa: E402


def card():
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=name,power.limit,clocks.max.sm",
                              "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clk = [s.strip() for s in out.split(",")]
        return dict(name=name, power_limit=power, max_sm_clock=clk)
    except Exception as e:                    # the timing itself does not depend on it
        return dict(name=torch.cuda.get_device_name(), power_limit=f"unavailable ({type(e).__name__})")


def run_leg(cfg_name, B, seconds, steps, warmup, segment_dur=None, overlap_ratio=None):
    cfg = get_config(cfg_name)
    dev = torch.device("cuda", torch.cuda.current_device())
    model = B200Encodec(cfg, init_state_dict(cfg, 0), str(dev), segment_dur=segment_dur, overlap_ratio=overlap_ratio)
    C, L, D = cfg.channels, int(seconds * cfg.sample_rate), cfg.dimension
    n_q = cfg.num_quantizers
    n_rot = max(2, int(140e6 // (B * C * L * 4)) + 1)
    g = torch.Generator().manual_seed(4800 + C)
    shape = (B, C, L) if C > 1 else (B, L)
    wavs = [(0.1 * torch.randn(shape, generator=g)).to(dev) for _ in range(n_rot)]
    recon = torch.empty((B, C, L), dtype=torch.float32, device=dev)
    if segment_dur is None:
        Tf = cfg.frames(L)
        codes = torch.empty((n_q, B, Tf), dtype=torch.int64, device=dev)
        quant = torch.empty((B, Tf, D), dtype=torch.float32, device=dev)
        scale = torch.empty((B,), dtype=torch.float32, device=dev)
        frames_per_step = B * Tf

        def step(i):
            model._ck(model._lib.fcb_roundtrip(model._h, _ptr(wavs[i % n_rot]), B, L, n_q, 1, _ptr(codes), _ptr(quant),
                                               _ptr(scale), None, _ptr(recon), model._stream()), "fcb_roundtrip")
    else:
        plan = model.plan_segments(L)
        codes = torch.empty(n_q * B * plan.total_frames, dtype=torch.int64, device=dev)
        quant = torch.empty(B * plan.total_frames * D, dtype=torch.float32, device=dev)
        scale = torch.empty(plan.n_seg * B, dtype=torch.float32, device=dev)
        frames_per_step = B * plan.total_frames

        def step(i):
            model._ck(model._lib.fcb_roundtrip_segmented(model._h, _ptr(wavs[i % n_rot]), B, L, model.segment_length,
                                                         model.segment_stride, n_q, 1, _ptr(codes), _ptr(quant), _ptr(scale),
                                                         _ptr(recon), model._stream()), "fcb_roundtrip_segmented")
    for i in range(max(warmup, 1)):
        t0 = time.perf_counter()
        step(i)
        torch.cuda.synchronize()
        print(f"{cfg_name} segment_dur={segment_dur}: warm-up step {i} {1e3 * (time.perf_counter() - t0):.1f} ms",
              file=sys.stderr, flush=True)
    print(f"{cfg_name} segment_dur={segment_dur}: timing {steps} steps", file=sys.stderr, flush=True)
    model.set_profiling(segment_dur is None)
    launches0 = model.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        step(warmup + i)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    res = dict(preset=cfg_name, B=B, seconds=seconds, channels=C, n_q=n_q, steps=steps, input_batches=n_rot,
               ms_per_step=round(ms / steps, 3), frames_per_s=round(frames_per_step * steps / (ms * 1e-3), 1),
               audio_s_per_s=round(B * seconds * steps / (ms * 1e-3), 1),
               launches_per_step=(model.launch_count() - launches0) / steps)
    if segment_dur is None:
        res["phase_ms_last_step"] = {k: round(v, 3) for k, v in model.phase_ms().items()}
        model.set_profiling(False)
    else:
        res.update(segment_dur=segment_dur, overlap_ratio=overlap_ratio, n_seg=plan.n_seg, n_full=plan.n_full,
                   n_tail=plan.n_tail)
    del model
    torch.cuda.synchronize()
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--batch", type=int, default=16)
    ap.add_argument("--seconds", type=float, default=10.0)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_stereo.py needs a CUDA device (there is no CPU path)")
    legs = dict(stereo_whole=run_leg("encodec_48k_stereo", args.batch, args.seconds, args.steps, args.warmup),
                stereo_segmented=run_leg("encodec_48k_stereo", args.batch, args.seconds, args.steps, args.warmup, 1.0, 0.01),
                mono_ds640=run_leg("encodec_16k_n32_ds640", args.batch, args.seconds, args.steps, args.warmup))
    print(json.dumps(dict(card=card(), legs=legs)))


if __name__ == "__main__":
    main()
