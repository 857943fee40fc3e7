#!/usr/bin/env python
"""bench.py -- codec frames/s (encode + RVQ + decode) on synthetic 16 kHz audio, BASELINE.json's metric.

    python bench.py --gpus N --steps K --warmup W          (N>1: launched by torch.distributed.run)
    python bench.py --impl reference ...                   (CPU arm: the oracle port of the reference path)

A "step" = one Encodec.inference-equivalent pass (RMS-normalise -> SEANet encoder -> 32-stage RVQ ->
SEANet decoder) over one batch.  Workload at N=1 = BASELINE.json configs[1]: encodec ds640, batch 16,
10 s clips, n_q=32.  For N>1 every rank processes its own 16 clips (weak scaling; clips are independent,
SURVEY.md §8(e)); the end-to-end number additionally scatters/gathers the clips over NCCL from rank 0.

Prints ONE JSON line (rank 0).  `value` = frames/s with inputs resident in HBM; `e2e` = the same metric through
the C-ABI host-buffer call (fcb_roundtrip_host: pinned host wav in, codes + recon out, copies inside).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (config, per-GPU batch, samples, bit_width)
    "config2": ("encodec_16k_n32_ds640", 16, 160000, None),
    "config1": ("encodec_16k_n32_ds640", 1, 160000, None),
    "config3": ("encodec_16k_n32_ds320", 64, 480000, None),
    "config5": ("encodec_16k_n32_ds640", 64, 160000, None),
    "config4": ("freqcodec_magphase_16k_n32_ds320", 32, 160000, None),
    # the grouped ("gr8") hub variant BASELINE config 4 names; its YAML is not in the repository (conv_group_ratio = 8 assumed
    # for the transposed convs too); the engine runs the grouped weights as dense block-diagonal matrices
    "config4_gr8": ("freqcodec_magphase_16k_n32_ds320_gr8", 32, 160000, None),
}
# roofline.traffic: dram__bytes_read.sum + dram__bytes_write.sum summed over the conv launches of ONE step
def load_ncu_traffic(workload):
    """profiles/conv_traffic.json = {workload: {"bytes": dram read + write of one step's conv launches, "source": file}},
    written by tools/summarize_ncu_raw.py from the latest `ncu --set full` capture (never a constant in this file)."""
    try:
        d = json.load(open(os.path.join(ROOT, "profiles", "conv_traffic.json")))
        e = d.get(workload)
        return (float(e["bytes"]), e.get("source")) if e else (None, None)
    except Exception:
        return (None, None)
# SURVEY.md §8(d) / BASELINE.md: algorithmic (layer-boundary) bytes and MACs per 10 s clip; re-derived analytically by
# funcodec_b200/workload.py and checked against it on CPU (tests/test_workload.py)
ALGO = {
    "encodec_16k_n32_ds640": dict(conv_bytes_per_10s=1066.6e6, conv_gmac_per_10s=33.10, lstm_gmac_per_10s=8.39,
                                  rvq_gflop_per_10s_nq32=2.10, weight_bytes=230.2e6),
    "freqcodec_magphase_16k_n32_ds320": dict(conv_bytes_per_10s=803.2e6, conv_gmac_per_10s=24.95, lstm_gmac_per_10s=4.20,
                                             rvq_gflop_per_10s_nq32=4.20, weight_bytes=64.9e6),
    # gr8: same activations; SURVEY §8(d): 10.42 GMAC per 10 s clip of grouped math (the engine executes the dense 24.95 and
    # reads the zero-expanded dense weights: 64.9 MB, where the grouped tensors themselves are 39.7 MB)
    "freqcodec_magphase_16k_n32_ds320_gr8": dict(conv_bytes_per_10s=803.2e6, conv_gmac_per_10s=10.42, lstm_gmac_per_10s=4.20,
                                                 rvq_gflop_per_10s_nq32=4.20, weight_bytes=64.9e6),
    "encodec_16k_n32_ds320": dict(conv_bytes_per_10s=780.1e6, conv_gmac_per_10s=15.67, lstm_gmac_per_10s=4.19,
                                  rvq_gflop_per_10s_nq32=4.19, weight_bytes=59.4e6),
}


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        # the conv / RVQ kernels are timed inside a long step: the SUSTAINED dense bf16 figure is the tensor denominator
        return dict(hbm_gbs=float(d["hbm_gbs"]), bf16_tflops=float(d.get("bf16_tflops_sustained", d.get("bf16_tflops", 0))),
                    source="measured")
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, source="fallback")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["unavailable"])
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return dict(sm_mhz=statistics.median(sm) if sm else None, sm_max_mhz=max(mx) if mx else None,
                    reasons=sorted(reasons), samples=len(sm))


def pick_cpu_threads(run_once):
    """ATen's CPU kernels for this path (small convs, LSTM steps) get SLOWER when oversubscribed (128 threads on the
    GPU box: 98 s per 10 s clip vs < 1 s with 16), so the baseline uses the fastest of a few thread counts."""
    import torch
    cores = os.cpu_count() or 1
    best, best_t = None, None
    for n in [c for c in (8, 16, 32, 64) if c <= cores] or [cores]:
        torch.set_num_threads(n)
        run_once()
        t0 = time.perf_counter()
        run_once()
        dt = time.perf_counter() - t0
        if best_t is None or dt < best_t:
            best, best_t = n, dt
        if dt > 4 * best_t:
            break
    torch.set_num_threads(best)
    return best


def make_oracle(cfg, sd, device="cpu"):
    """The CPU port of the reference model for this config (time-domain Encodec or mag_phase FreqCodec)."""
    if cfg.arch == 1:
        from oracle.freqcodec_oracle import OracleFreqCodec
        return OracleFreqCodec(sd, list(zip(cfg.ratios_f, cfg.ratios)), cfg.sample_rate, cfg.lstm_layers, cfg.n_fft, cfg.stft_hop)
    from oracle.encodec_oracle import OracleEncodec
    return OracleEncodec.from_config(sd, cfg, device=device)


def cpu_oracle_time(cfg, sd, B, L, bit_width, reps, warm):
    """Times the oracle (CPU port of the reference's PyTorch path) on a bounded sample; returns (frames/s, s/pass, threads)."""
    import torch
    o = make_oracle(cfg, sd)
    g = torch.Generator().manual_seed(1235)
    wav = 0.1 * torch.randn(B, L, generator=g)
    threads = pick_cpu_threads(lambda: o.inference(wav, need_recon=True, bit_width=bit_width, use_scale=True))
    ts = []
    for i in range(warm + reps):
        t0 = time.perf_counter()
        o.inference(wav, need_recon=True, bit_width=bit_width, use_scale=True)
        dt = time.perf_counter() - t0
        if i >= warm:
            ts.append(dt)
    med = statistics.median(ts)
    return B * cfg.frames(L) / med, med, threads


def run_reference(args):
    """--impl reference: the reference's CPU path (oracle port; /root/reference does not exist on the GPU box)."""
    import torch
    from funcodec_b200 import get_config, init_state_dict
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cfg_name, B, L, bw = WORKLOADS[args.workload]
    cfg = get_config(cfg_name)
    sd = init_state_dict(cfg, 0)
    # one step = the workload's own batch when a CPU pass of it fits the time budget (config 2: 16 x 10 s, ~6 s per pass on
    # 16 threads -> same_config), otherwise a bounded sample of ~2.56 M samples of audio per step
    sample_B = max(1, min(B, 2_560_000 // L))
    probe_B = min(sample_B, 2)
    o = make_oracle(cfg, sd)
    g = torch.Generator().manual_seed(1235)
    wav = 0.1 * torch.randn(sample_B, L, generator=g)

    def batched(n=None):
        o.inference(wav[:n or sample_B], need_recon=True, bit_width=bw)

    def per_clip(n=None):
        for i in range(n or sample_B):
            o.inference(wav[i:i + 1], need_recon=True, bit_width=bw)

    # give the CPU path its best configuration: fastest of {batched, clip-by-clip} x {8,16,32,64} threads, probed on 2 clips
    best = None
    for mode in (batched, per_clip):
        n = pick_cpu_threads(lambda: mode(probe_B))
        t0 = time.perf_counter()
        mode(probe_B)
        dt = time.perf_counter() - t0
        if best is None or dt < best[0]:
            best = (dt, mode, n)
    _, run_step, cores = best
    torch.set_num_threads(cores)
    for _ in range(args.warmup):
        run_step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        run_step()
    dt = time.perf_counter() - t0
    frames = sample_B * cfg.frames(L) * args.steps
    value = frames / dt
    what = "the full batch" if sample_B == B else f"bounded sample of batch {B}"
    sample = f"{sample_B} x {L / cfg.sample_rate:.0f} s clips per step ({run_step.__name__}; {what}), {cores} torch threads (fastest of 8/16/32/64 on {os.cpu_count()} host cores)"
    line = dict(metric="codec frames/sec (encode+RVQ+decode)", value=value, unit="frames/s", impl="reference",
                n_gpus=args.gpus, steps=args.steps, warmup=args.warmup, ms_per_step=1e3 * dt / args.steps,
                higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f32", data="synthetic",
                rtf=dt / (sample_B * L / cfg.sample_rate * args.steps),
                config=dict(workload=f"{cfg_name} B={B}/GPU L={L} n_q={cfg.num_quantizers_for_bandwidth(bw)} (BASELINE {args.workload})",
                            global_batch=args.gpus * B, clip_seconds=L / cfg.sample_rate, sample=sample,
                            same_config=bool(sample_B == B and args.gpus == 1)),
                cpu_baseline=dict(value=value, unit="frames/s", cores=cores, kind="port", sample=sample),
                e2e=dict(value=value, unit="frames/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0))
    print(json.dumps(line))


def config5_extra(model, cfg, dev, rank, world, steps=5):
    """BASELINE config 5 as named: ONE batch of 64 x world clips (10 s, ds640, n_q = 32) held by one process and sharded over
    the GPUs of the box.  Three timings (CUDA events, max over ranks): device-resident shards; end to end with the batch in
    a shared pinned host buffer that every rank DMA-reads / writes over its own PCIe link (parallel.SharedHostBatch, no
    data-path collective); end to end through rank 0's GPU with NCCL scatter / gather (parallel.ShardedCodec)."""
    import torch
    import torch.distributed as dist
    from funcodec_b200.encodec import _ptr
    from funcodec_b200.parallel import ShardedCodec, SharedHostBatch
    B, L = 64, 160000
    GB = world * B
    n_q, Tf = cfg.num_quantizers, cfg.frames(L)
    g = torch.Generator().manual_seed(4321 + rank)
    wavs = [(0.1 * torch.randn(B, L, generator=g)).to(dev) for _ in range(4)]      # 4 x 41 MB per rank > L2
    codes = torch.empty((n_q, B, Tf), dtype=torch.int64, device=dev)
    recon = torch.empty((B, 1, L), dtype=torch.float32, device=dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def run_dev(x):
        model._ck(model._lib.fcb_roundtrip(model._h, _ptr(x), x.shape[0], L, n_q, 1, _ptr(codes), None, None, None, _ptr(recon),
                                           model._stream()), "fcb_roundtrip")
        return codes, recon

    def timed(fn, n):
        for i in range(2):
            fn(i)
        torch.cuda.synchronize()
        dist.barrier()
        torch.cuda.synchronize()
        e0.record()
        for i in range(n):
            fn(2 + i)
        e1.record()
        torch.cuda.synchronize()
        dist.barrier()
        t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()) / n

    out = {}
    ms = timed(lambda i: run_dev(wavs[i % 4]), steps)
    out["device_resident"] = dict(ms_per_step=ms, frames_per_s=GB * Tf / (ms * 1e-3))
    # shared pinned host batch, one PCIe link per GPU (skipped, with the reason, when /dev/shm cannot hold the batch)
    shb, why = None, ""
    try:
        shb = SharedHostBatch(f"fcb_bench_{os.environ.get('MASTER_PORT', '0')}", GB, L, n_q, Tf, rank, world, create=(rank == 0))
    except OSError as exc:
        why = f"/dev/shm: {exc}"
    ok = torch.tensor([1 if shb is not None else 0], dtype=torch.int32, device=dev)
    dist.broadcast(ok, src=0)
    hw_host = hr_host = None
    if int(ok.item()) == 1:
        dist.barrier()
        shb.map()
        if rank == 0:
            shb.wav.copy_(0.1 * torch.randn(GB, L, generator=g))
        dist.barrier()
        lo, hi = shb.shard()
        ms = timed(lambda i: model.roundtrip_host(shb.wav[lo:hi], shb.codes[rank], shb.recon[lo:hi]), steps)
        out["e2e_shared_host"] = dict(ms_per_step=ms, frames_per_s=GB * Tf / (ms * 1e-3), h2d_bytes_per_step=GB * L * 4,
                                      d2h_bytes_per_step=n_q * GB * Tf * 8 + GB * L * 4,
                                      path="one /dev/shm batch page-locked by every rank; each rank fcb_roundtrip_host on its shard")
        hw_host, hr_host = shb.wav, shb.recon
    else:
        shb = None
        out["e2e_shared_host"] = dict(skipped=why or "rank 0 could not reserve the shared batch in /dev/shm")
    # NCCL scatter / gather through rank 0's GPU
    sharded = ShardedCodec(run_dev)
    hw = hc = hr = dw = None
    if rank == 0:
        hw = hw_host if hw_host is not None else (0.1 * torch.randn(GB, L, generator=g)).pin_memory()
        hc = torch.empty((n_q, GB, Tf), dtype=torch.int64).pin_memory()
        hr = hr_host if hr_host is not None else torch.empty((GB, 1, L), dtype=torch.float32).pin_memory()
        dw = torch.empty((GB, L), dtype=torch.float32, device=dev)

    def scatter_step(i):
        if rank == 0:
            dw.copy_(hw, non_blocking=True)
            o = sharded(dw, GB, L, dev)
            hc.copy_(o[0], non_blocking=True)
            hr.copy_(o[1], non_blocking=True)
        else:
            sharded(None, GB, L, dev)
        torch.cuda.synchronize()

    ms = timed(scatter_step, steps)
    out["e2e_nccl_scatter"] = dict(ms_per_step=ms, frames_per_s=GB * Tf / (ms * 1e-3),
                                   path="rank0 pinned host -> H2D -> NCCL scatter -> fcb_roundtrip -> NCCL gather -> D2H")
    out["workload"] = f"encodec_16k_n32_ds640 B={GB} ({B}/GPU) L={L} n_q={n_q} (BASELINE config 5 on {world} GPUs)"
    dist.barrier()
    if shb is not None:
        shb.close()
    return out


def cuda_eager_reference(cfg, sd, B, L, dev, reps=3):
    """Context only (BASELINE.md 'secondary comparison'): the oracle's torch functional restatement of the reference modules
    run on the SAME GPU in eager mode with TF32 off (cuDNN / cuBLAS fp32 kernels), device-resident input."""
    import torch
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    o = make_oracle(cfg, sd, device=dev)
    wav = 0.1 * torch.randn(B, L, device=dev)
    with torch.no_grad():
        o.inference(wav, need_recon=True)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            o.inference(wav, need_recon=True)
        e1.record()
        torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    return dict(ms_per_step=ms, frames_per_s=B * cfg.frames(L) / (ms * 1e-3), what="oracle (torch functional ops = the ATen/cuDNN "
                "kernels the reference modules call) on cuda, eager, allow_tf32=False, same batch; context, not the reference arm")


DUMP_LIMIT_BYTES = 63_000_000          # 64 MB with room for the .npy headers


def sample_outputs(outs, limit=DUMP_LIMIT_BYTES):
    """outs: {name: device tensor} of one step, clips on axis 1 for "codes" ([n_q, B, T]) and axis 0 otherwise -> {name: float32
    numpy array}.  Code indices are exact in float32.  When the whole batch exceeds `limit` bytes, the same fixed seeded sample
    of clips is taken from every array and its indices are returned as "clip_index"."""
    import torch
    axis = {name: 1 if name == "codes" else 0 for name in outs}
    B = outs["codes"].shape[1]
    per_clip = sum(t.numel() // t.shape[axis[n]] for n, t in outs.items()) * 4
    clips = None
    if B * per_clip > limit:
        keep = max(1, (limit - 8 * B) // per_clip)
        clips = torch.randperm(B, generator=torch.Generator().manual_seed(0))[:keep].sort().values
    res = {}
    for name, t in outs.items():
        t = t.detach().cpu()
        if clips is not None:
            t = t.index_select(axis[name], clips)
        res[name] = t.to(torch.float32).numpy()
    if clips is not None:
        res["clip_index"] = clips.to(torch.float32).numpy()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="config2", choices=sorted(WORKLOADS))
    ap.add_argument("--batch", type=int, default=0, help="override per-GPU batch")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--skip-e2e", action="store_true", help="profiling runs only (ncu): skip the host-buffer leg")
    ap.add_argument("--no-extras", action="store_true", help="skip the extra legs (config-5 block at N > 1, CUDA-eager context at N = 1)")
    ap.add_argument("--e2e-mode", choices=["sharded-host", "scatter"], default="sharded-host",
                    help="N > 1 end-to-end leg: every rank round-trips its own pinned host shard (default; the reference's "
                         "multi-process inference), or rank 0 holds the whole batch and scatters / gathers it over NCCL")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed on rank 0 (codes, quant, scale, recon) as DIR/<name>.npy in "
                         "float32; when they exceed 64 MB, a fixed seeded sample of clips (listed in DIR/clip_index.npy)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of --impl b200")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist
    from funcodec_b200 import get_config, init_state_dict
    from funcodec_b200.encodec import B200Encodec

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py --impl b200 needs a GPU (no CPU fallback)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    # stdout carries exactly ONE JSON line: everything else this process (and NCCL, whose NCCL_DEBUG the caller controls and
    # which logs to stdout) prints is routed to stderr by swapping the file descriptors; the line is written to the saved fd
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    cfg_name, B, L, bw = WORKLOADS[args.workload]
    if args.batch:
        B = args.batch
    cfg = get_config(cfg_name)
    sd = init_state_dict(cfg, 0)
    model = B200Encodec(cfg, sd, str(dev))
    n_q = cfg.num_quantizers_for_bandwidth(bw)
    Tf = cfg.frames(L)
    peaks = load_peaks()

    # inputs: rotate over enough distinct batches that consecutive steps never re-read an L2-resident input
    n_rot = max(2, int(140e6 // (B * L * 4)) + 1)
    g = torch.Generator().manual_seed(1234 + 2 + rank)
    wavs = [(0.1 * torch.randn(B, L, generator=g)).to(dev) for _ in range(n_rot)]
    codes = torch.empty((n_q, B, Tf), dtype=torch.int64, device=dev)
    quant = torch.empty((B, Tf, cfg.dimension), dtype=torch.float32, device=dev)
    scale = torch.empty((B, 1), dtype=torch.float32, device=dev)
    Lr = min(L, cfg.decoded_length(Tf))
    recon = torch.empty((B, 1, Lr), dtype=torch.float32, device=dev)
    import ctypes
    from funcodec_b200.encodec import _ptr

    def step(i):
        x = wavs[i % n_rot]
        if Lr == L:
            model._ck(model._lib.fcb_roundtrip(model._h, _ptr(x), B, L, n_q, 1, _ptr(codes), _ptr(quant), _ptr(scale),
                                               None, _ptr(recon), model._stream()), "fcb_roundtrip")
        else:   # FreqCodec clip whose iSTFT is shorter than L: encode + decode of what exists
            model._ck(model._lib.fcb_encode(model._h, _ptr(x), B, L, n_q, _ptr(codes), _ptr(quant), _ptr(scale), None, None,
                                            model._stream()), "fcb_encode")
            model._ck(model._lib.fcb_decode_emb(model._h, _ptr(quant), B, Tf, _ptr(scale), _ptr(recon), Lr, model._stream()),
                      "fcb_decode_emb")

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # clocks are sampled from before the warm-up (nvidia-smi needs ~0.3 s to start; the timed region of a short run
    # would otherwise be over before its first sample) -- same kernels, same load
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    for i in range(max(args.warmup, 3)):
        step(i)
    barrier()
    t_load = time.perf_counter()
    while rank == 0 and len(sampler.rows) < 2 and time.perf_counter() - t_load < 1.5:
        step(0)                     # keep the GPU under the same load until the sampler has started reporting
        torch.cuda.synchronize()
    barrier()

    # ---------------- timed region: device-resident inputs
    model.set_profiling(True)
    launches0 = model.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for i in range(args.steps):
        step(args.warmup + i)
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    launches = model.launch_count() - launches0
    phases = model.phase_ms()           # the last timed step's phase durations
    model.set_profiling(False)
    # later legs reuse these buffers: keep the last timed step's outputs now, write them at the end
    dumped = sample_outputs(dict(codes=codes, quant=quant, scale=scale, recon=recon)) if args.dump_outputs and rank == 0 else None
    clocks = sampler.stop() if rank == 0 else None
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = float(t.item())
    frames_total = world * B * Tf * args.steps
    value = frames_total / (ms_max * 1e-3)
    audio_s = world * B * L / cfg.sample_rate * args.steps

    # ---------------- end-to-end: host buffers through the C ABI (+ NCCL scatter/gather of clips for N>1)
    e2e_steps = max(3, min(args.steps, 10))
    e2e_ms, h2d, d2h = float("nan"), 0, 0
    if args.skip_e2e:
        pass
    elif world == 1 or args.e2e_mode == "sharded-host":
        # every rank owns its shard of the clips in ITS OWN pinned host memory and calls fcb_roundtrip_host on it: this is
        # the reference's multi-GPU inference (N processes over a split wav.scp, encoding_decoding.sh:69-100) -- the path
        # shards with no data-path collective
        hw = (0.1 * torch.randn(B, L, generator=g)).pin_memory()
        hc = torch.empty((n_q, B, Tf), dtype=torch.int64).pin_memory()
        hr = torch.empty((B, 1, L), dtype=torch.float32).pin_memory()
        for _ in range(2):
            model.roundtrip_host(hw, hc, hr)
        torch.cuda.synchronize()
        barrier()
        t0 = time.perf_counter()
        e0.record()
        for _ in range(e2e_steps):
            model.roundtrip_host(hw, hc, hr)
        e1.record()
        torch.cuda.synchronize()
        e2e_ms = max(e0.elapsed_time(e1), (time.perf_counter() - t0) * 1e3)
        barrier()
        if world > 1:
            t = torch.tensor([e2e_ms], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            e2e_ms = float(t.item())
        h2d = world * B * L * 4
        d2h = world * (hc.numel() * 8 + hr.numel() * 4)
    else:
        # --e2e-mode scatter: ONE in-memory batch held by rank 0 spread over the GPUs of the box (NCCL scatter / gather)
        from funcodec_b200.parallel import ShardedCodec
        GB = world * B

        def run_shard(w):
            model._ck(model._lib.fcb_roundtrip(model._h, _ptr(w), w.shape[0], L, n_q, 1, _ptr(codes), None, None, None,
                                               _ptr(recon), model._stream()), "fcb_roundtrip")
            return codes, recon

        sharded = ShardedCodec(run_shard)
        if rank == 0:
            hw = (0.1 * torch.randn(GB, L, generator=g)).pin_memory()
            hc = torch.empty((n_q, GB, Tf), dtype=torch.int64).pin_memory()
            hr = torch.empty((GB, 1, L), dtype=torch.float32).pin_memory()
            dw = torch.empty((GB, L), dtype=torch.float32, device=dev)

        def e2e_step():
            if rank == 0:
                dw.copy_(hw, non_blocking=True)
                out = sharded(dw, GB, L, dev)
                hc.copy_(out[0], non_blocking=True)
                hr.copy_(out[1], non_blocking=True)
            else:
                sharded(None, GB, L, dev)
            torch.cuda.synchronize()

        for _ in range(2):
            e2e_step()
        barrier()
        e0.record()
        for _ in range(e2e_steps):
            e2e_step()
        e1.record()
        barrier()
        t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_ms = float(t.item())
        h2d = GB * L * 4
        d2h = n_q * GB * Tf * 8 + GB * L * 4
    e2e_value = world * B * Tf * e2e_steps / (e2e_ms * 1e-3)

    extra = {}
    if not args.no_extras and not args.skip_e2e and not args.batch:
        try:
            if world > 1 and args.workload == "config2" and cfg.arch == 0:
                extra["config5"] = config5_extra(model, cfg, dev, rank, world)
            elif world == 1 and cfg.arch == 0:
                extra["reference_cuda_eager"] = cuda_eager_reference(cfg, sd, B, L, dev)
        except Exception as exc:            # an extra leg must never take the headline line down
            extra["error"] = f"{type(exc).__name__}: {exc}"

    if rank == 0:
        algo = ALGO[cfg_name]
        clip10 = L / 160000.0
        conv_ms = phases["encoder_conv"] + phases["decoder_conv"]
        conv_bytes = algo["conv_bytes_per_10s"] * clip10 * B + algo["weight_bytes"]
        achieved = conv_bytes / (conv_ms * 1e-3) / 1e9 if conv_ms > 0 else 0.0
        conv_tflops = 2 * algo["conv_gmac_per_10s"] * clip10 * B / (conv_ms * 1e-3) / 1e3 if conv_ms > 0 else 0.0
        traffic, traffic_src = load_ncu_traffic(args.workload) if not args.batch else (None, None)
        # tensor-pipe view (north_star: "tensor-pipe utilisation (RVQ distance)"): fp32-equivalent FLOPs x 3 passes of the split
        # operands, against the measured dense bf16/fp16 rate (conv: kind::f16) or half of it (RVQ: kind::tf32)
        f16_peak = peaks["bf16_tflops"]
        conv_tensor_tflops = 3 * conv_tflops
        rvq_ms = phases.get("rvq", 0.0)
        rvq_tflops = 3 * algo["rvq_gflop_per_10s_nq32"] * (n_q / 32.0) * clip10 * B / (rvq_ms * 1e-3) / 1e3 if rvq_ms > 0 else 0.0
        tensor = dict(conv=dict(achieved=conv_tensor_tflops, peak=f16_peak, unit="TFLOP/s", frac=conv_tensor_tflops / f16_peak if f16_peak else None,
                                note="3 kind::f16 MMAs per fp32-equivalent product (fp16 hi/lo split); peak = measured dense bf16"),
                      rvq=dict(achieved=rvq_tflops, peak=f16_peak / 2, unit="TFLOP/s", frac=rvq_tflops / (f16_peak / 2) if f16_peak else None,
                               kernel_ms_per_step=rvq_ms,
                               note="rvq_tc_kernel: 3 kind::tf32 MMAs per product; peak = measured dense bf16 / 2 (tf32 rate); "
                                    "includes the argmin / re-scoring / residual-update epilogues of all stages"))
        roofline = dict(bound="hbm", kernel="conv1d_tc_kernel<N> (+ conv1d_cl / conv1d_cout1 for the 3 layers that do not fit "
                                            "the tensor cores): all SEANet conv/convtr launches of one step = "
                                            "encoder_conv + decoder_conv phases",
                        achieved=achieved, peak=peaks["hbm_gbs"], unit="GB/s", frac=achieved / peaks["hbm_gbs"],
                        traffic=traffic, traffic_source=traffic_src,
                        peak_source=peaks["source"], algorithmic_bytes=conv_bytes,
                        kernel_ms_per_step=conv_ms, conv_fp32_tflops=conv_tflops, tensor=tensor)
        cpu = None
        if not args.no_cpu_baseline:
            v, sec, cores = cpu_oracle_time(cfg, sd, 1, 160000, None, reps=5, warm=1)
            cpu = dict(value=v, unit="frames/s", cores=cores, host_cores=os.cpu_count(), kind="port",
                       sample="1 x 10 s clip (BASELINE config 1), n_q=32, median of 5 after 1 warm-up; "
                              "oracle = torch-CPU restatement of the reference modules", seconds_per_pass=sec,
                       rtf=sec / 10.0)
        line = dict(metric="codec frames/sec (encode+RVQ+decode)", value=value, unit="frames/s", n_gpus=world,
                    steps=args.steps, warmup=args.warmup, ms_per_step=ms_max / args.steps, higher_is_better=True,
                    scaling="weak", vs_baseline=None, dtype="f32", data="synthetic", impl="b200",
                    rtf=(ms_max * 1e-3) / audio_s,
                    config=dict(workload=f"{cfg_name} B={B}/GPU L={L} n_q={n_q} (BASELINE {args.workload})",
                                global_batch=world * B, clip_seconds=L / cfg.sample_rate,
                                l2="inputs rotated over %d distinct batches (>126 MB); per-step activation traffic >> L2" % n_rot,
                                parallelism=f"dp{world} (independent clips per GPU)"),
                    clocks=clocks, gpu_launches=int(launches),
                    e2e=dict(value=e2e_value, unit="frames/s", h2d_bytes_per_step=int(h2d), d2h_bytes_per_step=int(d2h),
                             ms_per_step=e2e_ms / e2e_steps, steps=e2e_steps,
                             path="fcb_roundtrip_host (pinned host buffers, one shard per rank)"
                                  if (world == 1 or args.e2e_mode == "sharded-host") else
                                  "rank0 pinned host -> H2D -> NCCL scatter -> fcb_roundtrip -> NCCL gather -> D2H"),
                    roofline=roofline, cpu_baseline=cpu, phase_ms_last_step=phases, extra=extra,
                    reference_arm_note=("the --impl reference arm is ONE CPU process (rank 0) at every N: a ratio of this N-GPU "
                                        "aggregate to it scales with N by construction" if world > 1 else None))
        if dumped is not None:
            import numpy as np
            os.makedirs(args.dump_outputs, exist_ok=True)
            for name, arr in dumped.items():
                np.save(os.path.join(args.dump_outputs, name + ".npy"), arr)
        sys.stdout.flush()
        os.write(json_fd, (json.dumps(line) + "\n").encode())
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
