#!/usr/bin/env python
"""bench.py -- separated-audio-seconds per second of the Conv-TasNet path (forward + SI-SDR/PIT loss).

    python bench.py --gpus N --steps K --warmup W            # our sm_100a path (one process per GPU under torchrun)
    python bench.py --impl reference --steps K --warmup W    # the reference algorithm on the host CPU cores (oracle port)
    python bench.py --config cfg4                            # DPRNN-TasNet (segment / overlap-add path), its own line
    python bench.py --train [--n-sources 3 --batch 8]        # the training step alone, its own line
    python bench.py ... --dump-outputs DIR                   # also write what the last timed step returned, as DIR/<name>.npy

Workload (BASELINE.json configs[1], "cfg2"): Conv-TasNet N=512 L=16 B=128 H=512 Sc=128 P=3 X=8 R=3, gLN, 2 speakers,
batch 32 x 4 s @ 8 kHz per GPU (weak scaling: every rank gets its own batch of 32; no data-path collective).
A "step" = one pass of the hot path (model forward + PIT(NegSISDR) loss) over one batch of synthetic mixtures.
Prints ONE JSON line on rank 0:
  value  = device-resident throughput (stage timers OFF), max over ranks, CUDA events;
  e2e    = the same through the C-ABI host-buffer call (ctn_convtasnet_loss_host via ConvTasNet.separate_host): pinned host
           mixture + sources -> H2D -> forward + PIT -> D2H of the separated estimates, loss and permutation, every step;
  stages = per-kernel-group CUDA-event times from a SEPARATE short pass with the library's stage timers on;
  train  = the data-parallel TRAINING step at the cfg3 per-GPU shape (3 speakers, batch 8 per GPU): fwd + PIT + backward +
           ONE gradient all-reduce (timed on its own) + native clip/Adam -- the path that has a collective, at every N;
  ddp_check (N > 1) = all-reduced shard gradients vs the same global batch on one GPU (small model), worst relative error.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "dnn-based_source_separation_b200"))

PAPER = dict(n_basis=512, kernel_size=16, sep_hidden_channels=512, sep_bottleneck_channels=128, sep_skip_channels=128,
             sep_kernel_size=3, sep_num_blocks=3, sep_num_layers=8)
CFG4 = dict(n_basis=64, kernel_size=2, sep_hidden_channels=128, sep_bottleneck_channels=64, sep_chunk_size=250, sep_hop_size=125,
            sep_num_blocks=6)
METRIC = "audio-sec/s Conv-TasNet 2spk 4s@8kHz fwd+SI-SDR-PIT"
# CPU arm: fixed team size and mini-batch.  Round-1 sweeps on the GPU box's host (128 logical cores) found 8-16 torch threads on
# 4-mixture mini-batches fastest (the reference trainer's own batch size is 4); 32 threads on the whole 32-mixture batch is 2.4x slower.
CPU_THREADS = 16
CPU_CHUNK = 4


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="cfg2", choices=["cfg2", "cfg3", "cfg4", "cfg5"],
                    help="cfg2 (default, the headline), cfg3 = 3 speakers batch 8 per GPU, cfg5 = 4 speakers 8 s @ 16 kHz batch 16 per GPU, "
                         "cfg4 = DPRNN-TasNet batch 16")
    ap.add_argument("--batch", type=int, default=None, help="mixtures per GPU per step")
    ap.add_argument("--seconds", type=float, default=None)
    ap.add_argument("--sample-rate", type=int, default=None)
    ap.add_argument("--n-sources", type=int, default=None)
    ap.add_argument("--math", default=None, choices=[None, "fp32", "tf32x3", "tf32", "f16x3"])
    ap.add_argument("--cpu-batch", type=int, default=None, help="mixtures per CPU-arm step (default: the full per-GPU batch)")
    ap.add_argument("--no-lib-ab", action="store_true", help="cfg4: skip the A/B step on the library (cuDNN) recurrence")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-train-block", action="store_true")
    ap.add_argument("--train", action="store_true", help="time the TRAINING step only; prints its own line")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one returned as DIR/<name>.npy (rank 0; inputs are seeded, so two "
                         "builds run with the same arguments can be compared output for output)")
    a = ap.parse_args()
    if a.dump_outputs and a.impl == "reference":
        ap.error("--dump-outputs writes what the sm_100a path computed; it does not apply to --impl reference")
    d = {"cfg2": (32, 4.0, 8000, 2), "cfg3": (8, 4.0, 8000, 3), "cfg4": (16, 4.0, 8000, 2), "cfg5": (16, 8.0, 16000, 4)}[a.config]
    a.batch = a.batch if a.batch is not None else d[0]
    a.seconds = a.seconds if a.seconds is not None else d[1]
    a.sample_rate = a.sample_rate if a.sample_rate is not None else d[2]
    a.n_sources = a.n_sources if a.n_sources is not None else d[3]
    return a


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return dict(hbm=p["hbm_gbs"], bf16_burst=p["bf16_tflops"], bf16_sustained=p.get("bf16_tflops_sustained", p["bf16_tflops"]),
                    source="measured (MEASURED_PEAKS.json)")
    return dict(hbm=6650.0, bf16_burst=1590.0, bf16_sustained=1400.0, source="fallback (B200_PROFILING.md)")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.stop, self.th = index, [], threading.Event(), None

    def _nvml(self):
        """NVML handle of the GPU (by UUID when torch exposes it, else by index); None -> fall back to the nvidia-smi subprocess."""
        try:
            import pynvml
            pynvml.nvmlInit()
            h = None
            try:
                import torch
                uuid = str(torch.cuda.get_device_properties(self.index).uuid)
                h = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid if not uuid.startswith("GPU-") else uuid).encode())
            except Exception:
                h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            return pynvml, h
        except Exception:
            return None, None

    def _run(self):
        nv, h = self._nvml()
        while not self.stop.is_set():
            try:
                if nv is not None:   # in-process NVML: ~10 ms period, several samples inside a 100-ms timed region
                    sm = nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
                    mx = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
                    try:
                        pw = nv.nvmlDeviceGetPowerUsage(h) / 1000.0
                    except Exception:
                        pw = 0.0
                    try:
                        rs = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                    except Exception:
                        rs = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                    act = lambda bit: "Active" if rs & bit else "Not Active"
                    self.rows.append([str(sm), str(mx), str(pw), act(0x8), act(0x40), act(0x20), act(0x4)])
                    self.stop.wait(0.01)
                    continue
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            self.stop.wait(0.1)

    def __enter__(self):
        self.th = threading.Thread(target=self._run, daemon=True)
        self.th.start()
        return self

    def __exit__(self, *a):
        self.stop.set()
        self.th.join(timeout=6)

    def summary(self):
        sm, mx, reasons = [], 0.0, set()
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = max(mx, float(r[1]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons), "samples": len(sm)}


DUMP_BYTES = 60 * 2 ** 20   # data budget of --dump-outputs; the .npy headers fit in what is left of 64 MB


def dump_outputs(path, arrays):
    """Writes each tensor of `arrays` as <path>/<name>.npy: floating point as float32 (float64 stays float64), integers as float64
    (exact).  Smallest first, every array gets an equal share of what is left of DUMP_BYTES; one larger than its share keeps every
    k-th element of its flattened values, the same elements on every run."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    items = sorted(arrays.items(), key=lambda kv: kv[1].numel())
    left = DUMP_BYTES
    for i, (name, t) in enumerate(items):
        a = t.detach().cpu().numpy()
        a = a.astype(np.float64 if a.dtype == np.float64 or a.dtype.kind in "iub" else np.float32)
        share = max(1, left // (len(items) - i) // a.itemsize)
        if a.size > share:
            a = a.reshape(-1)[::-(-a.size // share)]
        np.save(os.path.join(path, name + ".npy"), a)
        left -= a.nbytes


def workload_config(args, world):
    """The `config` object of BOTH arms (ours and --impl reference): same keys, same values => same_config."""
    B, S = args.batch, args.n_sources
    if args.config == "cfg4":
        wl = (f"cfg4: DPRNN-TasNet {S}spk N64 L2 F64 H128 K250 P125 B6 gLN sigmoid, batch {B} x {args.seconds:g}s@{args.sample_rate // 1000}kHz per GPU, "
              "fwd + PIT(NegSISDR)")
    else:
        wl = (f"{args.config}: Conv-TasNet {S}spk N512 L16 B128 H512 Sc128 P3 X8 R3 gLN sigmoid, batch {B} x {args.seconds:g}s@"
              f"{args.sample_rate // 1000}kHz per GPU, fwd + PIT(NegSISDR)")
    return {"workload": wl, "global_batch": world * B,
            "l2": "per-step activation traffic (> 2 GB) exceeds the 126 MB L2 many times over; no explicit flush"}


# ---------------------------------------------------------------------------------------------------------------
def cpu_reference_leg(args, steps, warmup, cpu_batch):
    """The reference algorithm (oracle port, plain PyTorch CPU ops = the ATen ops the reference dispatches to) on the host cores,
    fixed team of CPU_THREADS torch threads, `cpu_batch` mixtures of the workload's shape per step."""
    import torch
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import convtasnet_oracle as O
    cores = os.cpu_count() or 1
    thr = min(CPU_THREADS, cores)
    torch.set_num_threads(thr)
    T = int(args.seconds * args.sample_rate)
    if args.config == "cfg4":
        import dprnn_oracle as DO
        cfg = DO.DPRNNConfig(**CFG4, n_sources=args.n_sources)
        sd = DO.synth_state_dict(cfg, seed=111)
        fwd = lambda m: DO.dprnn_tasnet_fwd(m, sd, cfg)
    else:
        cfg = O.OracleConfig(**PAPER, causal=False, n_sources=args.n_sources)
        sd = O.synth_state_dict(cfg, seed=111)
        fwd = lambda m: O.conv_tasnet_fwd(m, sd, cfg)
    mixture, sources = O.synth_batch(cpu_batch, args.n_sources, T, seed=111)
    times = []
    with torch.no_grad():
        for i in range(warmup + steps):
            t0 = time.perf_counter()
            tot = 0.0
            for lo in range(0, cpu_batch, CPU_CHUNK):     # one step = the whole batch, walked in mini-batches of CPU_CHUNK mixtures
                out, _ = fwd(mixture[lo:lo + CPU_CHUNK])
                loss_b, perm = O.pit_neg_sisdr(out, sources[lo:lo + CPU_CHUNK], batch_mean=False)
                tot += float(loss_b.sum())
            if i >= warmup:
                times.append(time.perf_counter() - t0)
    total = sum(times)
    value = cpu_batch * args.seconds * len(times) / total
    return dict(value=value, unit="audio-sec/s", cores=thr, kind="port",
                sample=f"{cpu_batch} x {args.seconds:g} s @ {args.sample_rate} Hz per step, {len(times)} steps (+{warmup} warm-up), "
                       f"oracle/ port of the reference forward + PIT under no_grad in mini-batches of {CPU_CHUNK}, {thr} torch threads on {cores} logical cores",
                ms_per_step=1e3 * total / len(times))


def stage_model(args, B, frames, T):
    """Algorithmic (bytes, flops) per kernel GROUP of each stage (DESIGN.md section 5): one group = one launch, except `prep`."""
    N, Bc, H, Sc, S = PAPER["n_basis"], PAPER["sep_bottleneck_channels"], PAPER["sep_hidden_channels"], PAPER["sep_skip_channels"], args.n_sources
    L = PAPER["kernel_size"]
    RX = PAPER["sep_num_blocks"] * PAPER["sep_num_layers"]
    f = frames * B * 4.0
    Mt = Bc + Sc
    return {
        "enc": (B * T * 4.0 + N * f, 2.0 * N * L * frames * B, "hbm"),
        "head": ((N + Bc) * f, 2.0 * N * Bc * frames * B, "tensor"),
        # pw1 reads x_prev and the previous block's r[:Bc], writes x and h
        "pw1": ((3 * Bc + H) * f, 2.0 * Bc * H * frames * B, "tensor"),
        "dw": (2.0 * H * f, 2.0 * 3 * H * frames * B, "hbm"),
        "pw2": ((H + Mt) * f, 2.0 * H * Mt * frames * B, "tensor"),
        # ONE launch: reads the skip rows of all RX blocks, writes the skip sum
        "fin": ((RX * Sc + Sc) * f, 2.0 * RX * Sc * frames * B, "hbm"),
        "mask": ((Sc + N + S * N) * f, 2.0 * Sc * S * N * frames * B, "tensor"),
        "dec": (S * N * f + S * B * T * 4.0, 2.0 * S * N * L * frames * B, "hbm"),
        "loss": (2 * 2.0 * S * B * T * 4.0 / 3.0, 0.0, "hbm"),   # 3 launches share two passes over est+tgt
        "prep": (0.0, 0.0, "hbm"),
    }


def cuda_time(fn, steps, torch, D, dev, sampler=None):
    """barrier + synchronize, EXACTLY `steps` calls between two CUDA events, synchronize + barrier; max over ranks (ms)."""
    D.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    ret = None
    for _ in range(steps):
        ret = fn()
    e1.record()
    torch.cuda.synchronize()
    D.barrier()
    ms_local = e0.elapsed_time(e1)
    return D.max_over_ranks(ms_local, dev), ms_local, ret


def build_convtasnet(args, dev, torch, S):
    from ctn_b200.models.conv_tasnet import ConvTasNet
    torch.manual_seed(111)  # reference default seed (train.sh:59); default init = the reference's default init
    m = ConvTasNet(PAPER["n_basis"], PAPER["kernel_size"], enc_basis="trainable", dec_basis="trainable", enc_nonlinear=None,
                   sep_hidden_channels=PAPER["sep_hidden_channels"], sep_bottleneck_channels=PAPER["sep_bottleneck_channels"],
                   sep_skip_channels=PAPER["sep_skip_channels"], sep_kernel_size=3, sep_num_blocks=3, sep_num_layers=8,
                   causal=False, n_sources=S).to(dev)
    m.math = args.math
    return m


def train_leg(args, torch, N, D, dev, rank, world, S, B, steps, warmup, outputs=None):
    """Data-parallel training step (egs/wsj0-mix/common/src/driver.py:146-157): fwd_train + PIT + native backward + ONE gradient
    all-reduce + native global-norm clip + Adam.  Returns the `train` block; fills `outputs`, if given, with the loss of the last
    timed step and the parameters it left (flattened, in named_parameters order)."""
    from ctn_b200.criterion.sdr import NegSISDR
    from ctn_b200.criterion.pit import PIT1d
    from ctn_b200.optim import FlatClipAdam
    T = int(args.seconds * args.sample_rate)
    model = build_convtasnet(args, dev, torch, S).train()
    crit = PIT1d(NegSISDR(), S)
    g = torch.Generator().manual_seed(211 + rank)
    sources = (0.1 * torch.randn(B, S, T, generator=g)).to(dev)
    mixture = sources.sum(dim=1, keepdim=True)
    opt = FlatClipAdam(model, lr=1e-3, max_norm=5.0)
    ar_ev = []

    def step():
        opt.zero_grad()
        loss, _ = crit(model(mixture), sources)
        loss.backward()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        nel = D.allreduce_gradients(model)
        e1.record()
        ar_ev.append((e0, e1))
        opt.step()
        return loss, nel

    for _ in range(max(warmup, 2)):
        loss, nel = step()
    launches = model.last_launches + model.last_bwd_launches + opt.launches_per_step
    ar_ev.clear()
    ms, _, (loss, nel) = cuda_time(step, steps, torch, D, dev)
    if outputs is not None:
        outputs["loss"] = loss.detach()
        outputs["params"] = torch.cat([p.detach().flatten() for p in model.parameters()])
    ar_ms = D.max_over_ranks(sum(a.elapsed_time(b) for a, b in ar_ev) / max(1, len(ar_ev)), dev)
    return {"workload": f"cfg3 per-GPU shape: Conv-TasNet {S}spk paper hparams, batch {B} x {args.seconds:g}s@{args.sample_rate // 1000}kHz per GPU, "
                        "fwd_train + PIT + backward + all-reduce + clip(5.0) + Adam(1e-3)", "global_batch": world * B,
            "ms_per_step": ms / steps, "allreduce_ms": ar_ms, "allreduce_elems": nel, "audio_s_per_s": world * B * args.seconds * steps / (ms * 1e-3),
            "steps": steps, "gpu_launches_per_step": launches, "optimizer": "native flat clip + Adam (ctn_clip_adam_step)",
            "peak_mem_gb": torch.cuda.max_memory_allocated(dev) / 1e9, "last_loss": float(loss.detach())}


def ddp_check(torch, D, dev, rank, world):
    """All-reduced shard gradients == gradients of the same GLOBAL batch on one GPU (small model; tests/test_dist_gpu.py)."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import convtasnet_oracle as O
    from ctn_b200.models.conv_tasnet import ConvTasNet
    from ctn_b200.criterion.sdr import NegSISDR
    from ctn_b200.criterion.pit import PIT1d
    cfg = O.OracleConfig(n_basis=32, kernel_size=16, sep_hidden_channels=64, sep_bottleneck_channels=32, sep_skip_channels=32,
                         sep_num_blocks=2, sep_num_layers=2, causal=False, n_sources=2)
    sd = O.synth_state_dict(cfg, seed=7)
    G = 3 * world
    mixture, sources = O.synth_batch(G, 2, 2000, seed=9)
    crit = PIT1d(NegSISDR(), 2)

    def grads(lo, hi):
        m = ConvTasNet(cfg.n_basis, cfg.kernel_size, enc_basis="trainable", dec_basis="trainable", enc_nonlinear=None,
                       sep_hidden_channels=cfg.sep_hidden_channels, sep_bottleneck_channels=cfg.sep_bottleneck_channels,
                       sep_skip_channels=cfg.sep_skip_channels, sep_num_blocks=cfg.sep_num_blocks, sep_num_layers=cfg.sep_num_layers,
                       causal=False, n_sources=2)
        m.load_state_dict(sd)
        m = m.to(dev).train()
        loss, _ = crit(m(mixture[lo:hi].to(dev)), sources[lo:hi].to(dev))
        loss.backward()
        return m

    lo, hi = D.shard_bounds(G, rank, world)
    m = grads(lo, hi)
    D.allreduce_gradients(m, local_batch=hi - lo, global_batch=G)
    full = grads(0, G)
    worst = 0.0
    for (k, p), (_, q) in zip(m.named_parameters(), full.named_parameters()):
        worst = max(worst, float((p.grad - q.grad).abs().max()) / (float(q.grad.abs().max()) + 1e-30))
    worst = D.max_over_ranks(worst, dev)
    return {"worst_rel": worst, "ok": bool(worst < 1e-4), "global_batch": G, "ranks": world,
            "what": "NCCL all-reduced shard gradients vs the same global batch on one GPU, all parameter tensors"}


def main():
    args = parse()
    if args.impl == "reference":
        rank = int(os.environ.get("RANK", "0"))
        if rank != 0:
            return
        world = int(os.environ.get("WORLD_SIZE", "1"))
        cpu_batch = args.cpu_batch or args.batch
        leg = cpu_reference_leg(args, args.steps, args.warmup, cpu_batch)
        cfgd = workload_config(args, max(world, args.gpus))
        line = {"impl": "reference", "metric": METRIC, "value": leg["value"], "unit": "audio-sec/s", "n_gpus": args.gpus,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": leg["ms_per_step"], "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": cfgd,
                "cpu_step": f"{cpu_batch} mixtures per CPU step" + ("" if cpu_batch == args.batch else f" (bounded sample of the batch-{args.batch} step)"),
                "cpu_baseline": {k: leg[k] for k in ("value", "unit", "cores", "kind", "sample")},
                "e2e": {"value": leg["value"], "unit": "audio-sec/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        print(json.dumps(line), flush=True)
        return

    import torch
    from ctn_b200 import _native as N
    from ctn_b200 import dist as D
    from ctn_b200.criterion.sdr import NegSISDR
    from ctn_b200.criterion.pit import PIT1d

    rank, local_rank, world = D.init()
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback); use --impl reference for the CPU arm"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    S, B, T = args.n_sources, args.batch, int(args.seconds * args.sample_rate)
    math_name = args.math or ("f16x3" if N.ctn_has_tcgen05() else "fp32")

    if args.train:
        outputs = {} if args.dump_outputs and rank == 0 else None
        blk = train_leg(args, torch, N, D, dev, rank, world, S, B, args.steps, args.warmup, outputs)
        if rank == 0:
            if outputs is not None:
                dump_outputs(args.dump_outputs, outputs)
            print(json.dumps({"mode": "train", "metric": "audio-sec/s Conv-TasNet TRAIN step", "value": blk["audio_s_per_s"], "unit": "audio-sec/s",
                              "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 2), "ms_per_step": blk["ms_per_step"],
                              "higher_is_better": True, "scaling": "weak", "dtype": math_name, "data": "synthetic", "config": {"workload": blk["workload"]},
                              "train": blk}), flush=True)
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()
        return

    if args.config == "cfg4":
        from ctn_b200.models.dprnn_tasnet import DPRNNTasNet
        torch.manual_seed(111)
        model = DPRNNTasNet(CFG4["n_basis"], CFG4["kernel_size"], enc_basis="trainable", dec_basis="trainable", enc_nonlinear=None,
                            sep_hidden_channels=CFG4["sep_hidden_channels"], sep_bottleneck_channels=CFG4["sep_bottleneck_channels"],
                            sep_chunk_size=CFG4["sep_chunk_size"], sep_hop_size=CFG4["sep_hop_size"], sep_num_blocks=CFG4["sep_num_blocks"],
                            causal=False, n_sources=S).to(dev).eval()
        model.math = args.math
    else:
        model = build_convtasnet(args, dev, torch, S).eval()
    crit = PIT1d(NegSISDR(), S)
    g = torch.Generator().manual_seed(111 + rank)
    sources_h = (0.1 * torch.randn(B, S, T, generator=g)).pin_memory()
    mixture_h = sources_h.sum(dim=1, keepdim=True).pin_memory()
    out_h = torch.empty(B, S, T).pin_memory()
    mixture_d, sources_d = mixture_h.to(dev), sources_h.to(dev)

    def step_resident():
        out = model(mixture_d)
        loss, perm = crit(out, sources_d)
        return out, loss, perm

    if args.config == "cfg4":
        loss_pin = torch.empty(1).pin_memory()
        perm_pin = torch.empty(B, S, dtype=torch.int64).pin_memory()

        def step_e2e():
            out = model(mixture_h.to(dev, non_blocking=True))
            loss, perm = crit(out, sources_h.to(dev, non_blocking=True))
            out_h.copy_(out, non_blocking=True)
            loss_pin.copy_(loss.reshape(1), non_blocking=True)
            perm_pin.copy_(perm, non_blocking=True)
            torch.cuda.current_stream().synchronize()
            return float(loss_pin[0])
        e2e_api = "DPRNNTasNet.forward + PIT1d(NegSISDR).forward on pinned host tensors, estimates + loss + permutation copied back"
    else:
        def step_e2e():
            loss, perm = model.separate_host(mixture_h, sources_h, out_host=out_h)
            torch.cuda.current_stream().synchronize()   # the caller reads the estimates / loss every step (driver.py:157 loss.item())
            return float(loss[0])
        e2e_api = ("ConvTasNet.separate_host -> ctn_convtasnet_loss_host (C ABI, host buffers): H2D mixture + sources, forward + PIT, "
                   "D2H estimates + loss + permutation")

    with torch.no_grad():
        for _ in range(max(args.warmup, 3)):
            step_resident()
        launches_per_step = getattr(model, "last_launches", 0) + N.ctn_last_launch_count()
        if args.config == "cfg4":   # the DPRNN path is made of many entry calls: count one whole step
            n0 = N.ctn_total_launch_count()
            step_resident()
            launches_per_step = int(N.ctn_total_launch_count() - n0)
        torch.cuda.synchronize()
        # ---- timed: device-resident, stage timers OFF ---------------------------------------------------------
        N.ctn_profile_enable(0)
        with ClockSampler(local_rank) as clk:
            ms, ms_local, last = cuda_time(step_resident, args.steps, torch, D, dev)
        outputs = None
        if args.dump_outputs and rank == 0:   # copied now: the calls below may reuse the device buffers
            outputs = {name: t.cpu() for name, t in zip(("estimates", "loss", "perm"), last)}
        # ---- timed: end to end ----------------------------------------------------------------------------------
        for _ in range(2):
            step_e2e()
        ms_e2e, _, last_loss = cuda_time(step_e2e, args.steps, torch, D, dev)
        # ---- stage pass (separate, not part of `value`) ------------------------------------------------------------
        prof, prof_steps, ms_prof = {}, min(args.steps, 5), 0.0
        if args.config != "cfg4":
            N.ctn_profile_enable(1)
            N.profile_read()
            _, ms_prof, _ = cuda_time(step_resident, prof_steps, torch, D, dev)
            prof = N.profile_read()
            N.ctn_profile_enable(0)

    train_blk, ddp = None, None
    if args.config == "cfg2" and not args.no_train_block:
        torch.cuda.empty_cache()
        N.release_workspaces()
        try:
            train_blk = train_leg(args, torch, N, D, dev, rank, world, 3, 8, steps=min(args.steps, 10), warmup=2)
        except Exception as e:  # the forward line must survive a failure of the auxiliary block
            train_blk = {"error": repr(e)[:300]}
        if world > 1:
            try:
                ddp = ddp_check(torch, D, dev, rank, world)
            except Exception as e:
                ddp = {"error": repr(e)[:300], "ok": False}

    audio_per_step = world * B * args.seconds
    value = audio_per_step * args.steps / (ms * 1e-3)
    e2e_value = audio_per_step * args.steps / (ms_e2e * 1e-3)
    if rank != 0:
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()
        return

    pk = peaks()
    frames = N.frames_of(T, model.kernel_size, model.stride)[0]
    tf32_peak = pk["bf16_sustained"] / (1.0 if math_name == "f16x3" else 2.0)
    stages, roof = {}, None
    if args.config != "cfg4":
        model_bf = stage_model(args, B, frames, T)
        for name, (t_ms, n) in prof.items():
            if n == 0:
                continue
            by, fl, bound = model_bf[name]
            groups = max(1, {"pw1": 24, "dw": 24, "pw2": 24}.get(name, 1) * prof_steps)
            per_group_ms = t_ms / groups
            ent = {"ms_per_step": t_ms / prof_steps, "launches_per_step": n / prof_steps, "share": t_ms / (ms_prof + 1e-9), "bound": bound,
                   "avg_launch_ms": t_ms / n}
            if by > 0:
                ent["GBps"] = by / (per_group_ms * 1e-3) / 1e9
                ent["hbm_frac"] = ent["GBps"] / pk["hbm"]
            if fl > 0 and bound == "tensor":
                ent["TFLOPs"] = fl / (per_group_ms * 1e-3) / 1e12
                ent["tensor_frac"] = ent["TFLOPs"] / tf32_peak
            stages[name] = ent
        dom = max((k for k in stages if k != "prep"), key=lambda k: stages[k]["ms_per_step"])
        d = stages[dom]
        traffic = None
        tpath = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tpath):
            traffic = json.load(open(tpath)).get(math_name, {}).get(dom)
        if d["bound"] == "tensor":
            roof = {"kernel": dom, "bound": "tensor", "achieved": d["TFLOPs"], "peak": tf32_peak, "unit": "TFLOP/s", "frac": d["TFLOPs"] / tf32_peak,
                    "traffic": traffic,
                    "peak_note": (f"fp16 dense = bf16_tflops_sustained of {pk['source']}" if math_name == "f16x3" else
                                  f"TF32 dense = bf16_tflops_sustained/2 of {pk['source']}") +
                                 "; algorithmic 2*M*N*K flops (the 3-pass hi/lo split issues 3x that on the tensor pipe)",
                    "hbm_view": {"achieved": d.get("GBps"), "peak": pk["hbm"], "unit": "GB/s", "frac": d.get("hbm_frac")}}
        else:
            roof = {"kernel": dom, "bound": "hbm", "achieved": d["GBps"], "peak": pk["hbm"], "unit": "GB/s", "frac": d["GBps"] / pk["hbm"],
                    "traffic": traffic, "peak_note": f"hbm_gbs of {pk['source']}"}
        # whole step against both roofs (SURVEY.md 8d: 234.3 MB and 39.28 GFLOP per 4-s 2-speaker sample, ideal fusion)
        step_bytes = sum(model_bf[k][0] * {"pw1": 24, "pw2": 24}.get(k, 1) for k in ("enc", "head", "pw1", "pw2", "fin", "mask", "dec"))
        roof["step"] = {"ms": ms / args.steps, "moved_bytes_model": step_bytes,
                        "hbm_frac_on_moved_bytes": step_bytes / (ms / args.steps * 1e-3) / 1e9 / pk["hbm"]}
    else:
        # cfg4: the step is 12 bi-LSTM + projection calls (tcgen05 kernel, csrc/ctn_lstm.cu) plus HBM-bound glue (segment, overlap-add,
        # gLN + residual + path swap).  Dominant kernel = the LSTM: timed alone here at the intra-chunk shape of the step.
        from ctn_b200.models import dprnn as dprnn_mod
        F_, K_, P_, H_ = CFG4["sep_bottleneck_channels"], CFG4["sep_chunk_size"], CFG4["sep_hop_size"], CFG4["sep_hidden_channels"]
        Sn = (frames + ((P_ - (frames - K_) % P_) % P_) - K_) // P_ + 1
        state = B * Sn * K_ * F_ * 4.0
        glue_bytes = 12 * 5 * state + 2 * state + 2 * B * F_ * frames * 4.0   # 12 x (P0,P1 read twice... see DESIGN 4.7) + segment + overlap-add
        blk = model.separator.dprnn.net[0].intra_chunk_block
        z = torch.randn(B * Sn, K_, F_, device=dev)
        Pbuf = torch.empty(2, B * Sn, K_, F_, device=dev)
        r_ = blk.rnn
        ptrs = (N._fp * 8)(*[t_.data_ptr() for t_ in (r_.weight_ih_l0, r_.weight_hh_l0, r_.bias_ih_l0, r_.bias_hh_l0, r_.weight_ih_l0_reverse,
                                                        r_.weight_hh_l0_reverse, r_.bias_ih_l0_reverse, r_.bias_hh_l0_reverse)])
        nws = N.ctn_bilstm_workspace_bytes(F_, H_, F_)
        wsb = torch.empty(max(nws, 16), dtype=torch.uint8, device=dev)

        def lstm_call():
            N.check(N.ctn_bilstm_proj_fwd(z.data_ptr(), B * Sn, K_, F_, H_, ptrs, blk.fc.weight.data_ptr(), F_, Pbuf.data_ptr(), None, None, wsb.data_ptr(),
                                          nws, N.stream_ptr(dev)), "ctn_bilstm_proj_fwd")
        native = bool(dprnn_mod.NATIVE_LSTM and N.ctn_bilstm_supported(F_, H_, F_))
        if native:
            for _ in range(3):
                lstm_call()
            ms_lstm, _, _ = cuda_time(lstm_call, 10, torch, D, dev)
            ms_lstm /= 10
            flops = 2.0 * (B * Sn) * K_ * (2.0 * (F_ + H_) * 4 * H_ + 2.0 * H_ * F_)   # both directions: gates + projection
            ach = flops / (ms_lstm * 1e-3) / 1e12
            # A/B: the same step with the library recurrence (cuDNN LSTM in IEEE fp32 + library GEMM for the Linear)
            ms_lib = float("nan")
            if not args.no_lib_ab:
                dprnn_mod.NATIVE_LSTM = False
                try:
                    with torch.no_grad():
                        step_resident()
                        ms_lib, _, _ = cuda_time(step_resident, 2, torch, D, dev)
                finally:
                    dprnn_mod.NATIVE_LSTM = True
            roof = {"kernel": "k_bilstm_pair (bi-LSTM recurrence + 2H->F projection, 2-CTA clusters, h in tensor memory; 12 calls per step)",
                    "bound": "tensor", "achieved": ach, "peak": tf32_peak, "unit": "TFLOP/s", "frac": ach / tf32_peak, "traffic": None,
                    "ms_per_call": ms_lstm, "algorithmic_flops_per_call": flops,
                    "peak_note": "fp16 dense = bf16_tflops_sustained of measured (MEASURED_PEAKS.json); algorithmic flops (the 3-pass hi/lo split issues "
                                 "3x that); a recurrence: 250 dependent steps per call, " + str(4 * ((B * Sn + 127) // 128)) + " CTAs",
                    "glue_bytes_per_step": glue_bytes, "glue_ideal_ms_at_peak": glue_bytes / (pk["hbm"] * 1e9) * 1e3,
                    "library_lstm_ms_per_step": (ms_lib / 2 if ms_lib == ms_lib else None), "native_lstm_ms_per_step": ms / args.steps,
                    "note": "library_lstm_ms_per_step = the same step with cuDNN's LSTM (IEEE fp32, as parity with the reference needs) + a library GEMM"}
        else:
            roof = {"kernel": "cuDNN LSTM (library)", "bound": "tensor", "achieved": None, "peak": tf32_peak, "unit": "TFLOP/s", "frac": None, "traffic": None}

    line = {
        "metric": METRIC if args.config == "cfg2" else METRIC.replace("Conv-TasNet 2spk 4s@8kHz", workload_config(args, world)["workload"].split(",")[0]),
        "value": value, "unit": "audio-sec/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": {"fp32": "f32 (CUDA-core FFMA)", "tf32x3": "f32 via 3xTF32 split on tcgen05, fp32 accumulate", "tf32": "tf32 (single pass), fp32 accumulate",
                  "f16x3": "f32 via 3xFP16 split on tcgen05 (kind::f16), fp32 accumulate"}[math_name],
        "data": "synthetic", "config": workload_config(args, world),
        "detail": {"math": math_name, "parallelism": f"batch shards x{world}, no data-path collective in the forward",
                   "value_timing": "CUDA events, stage timers off, max over ranks"},
        "e2e": {"value": e2e_value, "unit": "audio-sec/s", "h2d_bytes_per_step": B * T * 4 * (1 + S), "d2h_bytes_per_step": B * S * T * 4 + 4 + B * S * 8,
                "ms_per_step": ms_e2e / args.steps, "api": e2e_api},
        "gpu_launches": launches_per_step * args.steps,
        "roofline": roof, "stages": stages, "clocks": clk.summary(), "last_loss": last_loss,
    }
    if train_blk is not None:
        line["train"] = train_blk
    if ddp is not None:
        line["ddp_check"] = ddp
    if world == 1 and not args.no_cpu_baseline:
        # bounded sample: the full per-GPU batch, 1 warm-up + 2 timed steps (~ 20-30 s of CPU work at cfg2)
        leg = cpu_reference_leg(args, steps=2, warmup=1, cpu_batch=args.cpu_batch or args.batch)
        line["cpu_baseline"] = {k: leg[k] for k in ("value", "unit", "cores", "kind", "sample")}
    if outputs is not None:
        dump_outputs(args.dump_outputs, outputs)
    print(json.dumps(line), flush=True)
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
