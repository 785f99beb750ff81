#!/usr/bin/env python
"""bench.py — upstream frames/s of the B200 hot path (BASELINE.json metric) and the reference-CPU arm.

    python bench.py [--gpus N] [--steps K] [--warmup W]            # our arm (sm_100a kernels through the C ABI)
    python bench.py --impl reference [--steps K] [--warmup W]      # CPU arm: the reference itself on the host cores
    python bench.py --config {c1_fbank,c2,c3,c3_ll60k,c4}          # the other BASELINE.json configs (default c2)
    torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N   # N > 1: one rank per GPU over NCCL

Workload (BASELINE.json configs[1]): hubert_base (12L, 768d), global batch 32 x 10 s of synthetic 16 kHz audio
(seeded N(0,1) samples, fabricated random-init checkpoint — no network for data or weights). A "step" is one
pass of the hot path over the batch: UpstreamExpert(wavs) -> 13 hidden states [B, 499, 768] fp32 materialised,
then the Featurizer weighted sum; with N > 1 the batch is sharded by utterance (strong scaling, Lmax shared) and
the step ends with ONE NCCL all-gather of the weighted-sum features (SURVEY.md §8(e)).

One JSON line on stdout (rank 0). Keys beyond the base contract: "roofline" (tcgen05 GEMM kernel, algorithmic
FLOP/s from CUDA events around every GEMM launch in a profiled pass of the same steps), "cpu_baseline"
(oracle port on a bounded sample, rank 0, N=1), "e2e" (same metric through s3b_forward_host: pinned host
waveforms in, all hidden states back to pinned host memory, copies inside the timed region), "clocks".

    python bench.py ... --dump-outputs DIR

also writes, from rank 0, what the last timed step returned as float32 .npy files (see dump_outputs): features.npy
(the weighted sum, or the fbank features) and hidden_states.npy (every layer). Inputs and weights are seeded, so two
builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

SAMPLE_RATE = 16000
# BASELINE.json configs. c2 is the headline (the driver's default line); the others are selected with --config and
# their lines are committed under profiles/ (r2_bench_<config>.json).
CONFIGS = {
    "c2": dict(model="hubert_base", batch=32, seconds=10),
    "c3": dict(model="wav2vec2_large_960", batch=16, seconds=20),
    "c3_ll60k": dict(model="wav2vec2_large_ll60k", batch=16, seconds=20),
    "c4": dict(model="wavlm_base_plus", batch=32, seconds=10),
    "c1_fbank": dict(model="fbank", batch=4, seconds=1),
}


def metric_name(cfg_key: str) -> str:
    c = CONFIGS[cfg_key]
    if cfg_key == "c2":
        return "upstream frames/sec (16 kHz) hubert_base @ batch=32x10 s"  # BASELINE.json's metric, verbatim
    return f"upstream frames/sec (16 kHz) {c['model']} @ batch={c['batch']}x{c['seconds']} s"


def algorithmic_flops_per_utt(cfg, L):
    """SURVEY.md §8(d): conv + proj + posconv + linear + attn on the true frame count (multiply-add = 2)."""
    convs = [(512, 10, 5)] + [(512, 3, 2)] * 4 + [(512, 2, 2)] * 2
    n, cin, conv = L, 1, 0.0
    for dim, k, s in convs:
        n = (n - k) // s + 1
        conv += 2.0 * cin * dim * k * n
        cin = dim
    T, D, F, NL = n, cfg.encoder_embed_dim, cfg.encoder_ffn_embed_dim, cfg.encoder_layers
    proj = 2.0 * 512 * D * T
    pos = 2.0 * D * (D // cfg.conv_pos_groups) * cfg.conv_pos * T
    lin = NL * (8.0 * D * D + 4.0 * D * F) * T
    attn = NL * 4.0 * T * T * D
    return conv + proj + pos + lin + attn, T


def gemm_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum per GEMM launch (average over the launches of one step) from the
    committed ncu capture of `tools/profile_step.py` (profiles/r2_traffic.json, else round 1's; see profiles/README.md)."""
    for name in ("r2_traffic.json", "r1_traffic.json"):
        try:
            t = json.loads((ROOT / "profiles" / name).read_text())
            fam = [v for k, v in t.items() if k.startswith("gemm")]
            n = sum(v["launches"] for v in fam)
            if n:
                return sum(v["dram_bytes_per_launch"] * v["launches"] for v in fam) / n
        except Exception:
            continue
    return None


def seeded_wav(idx: int, n: int):
    import torch

    g = torch.Generator().manual_seed(1000 + idx)
    return torch.randn(n, generator=g)


DUMP_BYTES = 64 * 10**6  # --dump-outputs writes at most this many bytes in all (npy headers included)
NPY_HEADER = 128


def dump_outputs(out_dir: str, outputs: dict) -> None:
    """Write each output as out_dir/<name>.npy (float32). An output is a [B, T, D] tensor, or a sequence of them
    written stacked as [N, B, T, D]. Each output may use an equal share of DUMP_BYTES, plus whatever the outputs before
    it left unused. One larger than its share keeps a fixed sample of its B * T frames instead, [(N,) k, D]: the first
    k of torch.randperm(B * T) under seed 0, in ascending order. Their flat indices b * T + t go to
    out_dir/<name>_frames.npy (float64)."""
    import numpy as np
    import torch

    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    left = DUMP_BYTES
    for i, (name, x) in enumerate(outputs.items()):
        share = left // (len(outputs) - i)
        layers = list(x) if isinstance(x, (list, tuple)) else [x]
        B, T, D = layers[0].shape
        frame_bytes = len(layers) * D * 4
        if NPY_HEADER + B * T * frame_bytes > share:
            k = (share - 2 * NPY_HEADER) // (frame_bytes + 8)
            idx = torch.randperm(B * T, generator=torch.Generator().manual_seed(0))[:k].sort().values
            np.save(out / f"{name}_frames.npy", idx.double().numpy())
            left -= (out / f"{name}_frames.npy").stat().st_size
            layers = [h.reshape(B * T, D)[idx.to(h.device)] for h in layers]
        arr = torch.stack([h.float().cpu() for h in layers]).numpy()
        np.save(out / f"{name}.npy", arr if isinstance(x, (list, tuple)) else arr[0])
        left -= (out / f"{name}.npy").stat().st_size


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "25", "-i", str(self.index)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True,
            )
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def mark_begin(self):
        self.t0 = time.time()

    def stop(self):
        """Summary of the samples taken between mark_begin() and now (the timed + profiled passes)."""
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        t1 = time.time()
        time.sleep(0.05)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, power = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ts, ln in self.lines:
            if ts < getattr(self, "t0", 0.0) or ts > t1 + 0.03:
                continue
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[0])), mx.append(float(f[1])), power.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(names, f[4:8]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {
            "sm_mhz": sm[len(sm) // 2] if sm else None,
            "sm_max_mhz": max(mx) if mx else None,
            "power_w_max": max(power) if power else None,
            "samples": len(sm),
            "reasons": sorted(reasons),
        }


def usable_cores() -> int:
    """Host cores this process may really use: min(affinity mask, cgroup v2/v1 CPU quota). On the GPU boxes
    os.cpu_count() reports 128 while the container is capped at 16 CPUs; 128 threads would thrash."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = Path("/sys/fs/cgroup/cpu.max").read_text().split()[:2]
        if quota != "max":
            n = min(n, max(1, int(int(quota) / int(period))))
    except Exception:
        try:
            q = int(Path("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read_text())
            p = int(Path("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read_text())
            if q > 0:
                n = min(n, max(1, q // p))
        except Exception:
            pass
    return n


def cpu_arm(cfg_key: str, n_utts: int, steps: int, warmup: int, budget_s: float = None):
    """Time the reference's CPU implementation of the step on `n_utts` utterances of the workload, all usable host
    threads. kind = "reference": the UNMODIFIED reference (s3prl UpstreamExpert + Featurizer from the checkout beside this
    repository or S3PRL_REFERENCE, else the oracle/_ref install, oracle/build_ref.py) on the fabricated checkpoint; kind = "port": the oracle restatement
    (only when the reference is not present). Returns (frames/s, ms/step, cores, kind, steps actually timed)."""
    import torch

    sys.path.insert(0, str(ROOT / "oracle"))
    c = CONFIGS[cfg_key]
    cores = usable_cores()
    torch.set_num_threads(cores)
    L = c["seconds"] * SAMPLE_RATE
    wavs = [seeded_wav(i, L) for i in range(n_utts)]
    import ref_runtime as R

    if c["model"] == "fbank":
        if R.reference_root() is not None:
            R.activate()
            from s3prl.upstream.baseline.hubconf import fbank as ref_fbank

            expert, kind = ref_fbank(), "reference"
            expert.eval()
            run = lambda: expert(wavs)["hidden_states"][0]
        else:
            import fbank_oracle as FO

            kind = "port"
            run = lambda: FO.fbank_forward(wavs)
    else:
        from s3prl_b200.upstream.configs import get_arch
        from s3prl_b200.upstream.weights import fabricate_state_dict

        cfg = get_arch(c["model"])
        sd = fabricate_state_dict(cfg, seed=0)
        if R.reference_root() is not None:
            expert = R.reference_expert(c["model"], sd)
            feat = R.reference_featurizer(expert)
            kind = "reference"

            def run():
                return torch.nn.utils.rnn.pad_sequence(feat(wavs, expert(wavs)), batch_first=True)
        else:
            import upstream_oracle as O

            w = torch.zeros(cfg.encoder_layers + 1)
            kind = "port"

            def run():
                hs, _ = O.upstream_forward(wavs, sd, cfg)
                return O.weighted_sum(hs, w)

    times, frames = [], 0
    t_begin = time.perf_counter()
    with torch.no_grad():
        for it in range(warmup + steps):
            t0 = time.perf_counter()
            out = run()
            dt = time.perf_counter() - t0
            frames = out.shape[0] * out.shape[1]
            if it >= warmup:
                times.append(dt)
            # bounded: stop early (never before one timed step) when the wall-clock budget is spent
            if budget_s is not None and times and time.perf_counter() - t_begin > budget_s:
                break
    total = sum(times)
    return frames * len(times) / total, 1e3 * total / len(times), cores, kind, len(times)


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the step on this box's host cores, on the same
    config / metric / unit as our arm. Every step is the WHOLE batch of the config (same_config); the run is bounded to
    ~10 minutes of wall clock (it reports the steps it actually timed if it had to stop early)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    c = CONFIGS[args.config]
    fps, ms, cores, kind, timed = cpu_arm(args.config, c["batch"], args.steps, min(args.warmup, 2), budget_s=600.0)
    what = "the reference itself (s3prl UpstreamExpert + Featurizer, torch-CPU fp32)" if kind == "reference" else \
        "oracle port of the reference forward (reference not installed), torch-CPU fp32"
    sample = f"all {c['batch']} utterances x {c['seconds']} s per step; {what}, {cores} threads; {timed} timed steps"
    line = {
        "impl": "reference",
        "metric": metric_name(args.config), "value": fps, "unit": "frames/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(args.config, 1), "sample": sample, "steps_timed": timed},
        "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def workload_name(cfg_key: str, world: int) -> str:
    c = CONFIGS[cfg_key]
    if c["model"] == "fbank":
        return f"fbank upstream (80 log-mel + deltas + CMVN), batch {c['batch']} x {c['seconds']} s @16 kHz"
    per = c["batch"] // world
    return (f"{c['model']} forward + featurizer weighted sum, global batch {c['batch']} x {c['seconds']} s @16 kHz"
            + (f", sharded {per}/GPU + 1 all-gather of the weighted sum" if world > 1 else ""))


def run_fbank(args):
    """BASELINE config C1: fbank on 4 x 1 s (latency-bound: 392 frames). HBM roofline on the algorithmic bytes."""
    import torch

    from s3prl_b200 import hub

    c = CONFIGS[args.config]
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    L = c["seconds"] * SAMPLE_RATE
    wavs_host = [seeded_wav(i, L).pin_memory() for i in range(c["batch"])]
    wavs = [w.to(dev) for w in wavs_host]
    expert = hub.fbank().to(dev)
    sampler = ClockSampler(0)
    sampler.start()
    flush = torch.empty(256 * 1024 * 1024 // 4, device=dev)  # > 126 MB L2, rewritten between timed iterations
    with torch.no_grad():
        for _ in range(max(args.warmup, 3)):
            out = expert(wavs)["hidden_states"][0]
        torch.cuda.synchronize()
        sampler.mark_begin()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
        for a, b in ev:
            flush.zero_()
            a.record()
            out = expert(wavs)["hidden_states"][0]
            b.record()
        torch.cuda.synchronize()
        ms_step = sum(a.elapsed_time(b) for a, b in ev) / args.steps
        host_out = torch.empty(out.shape, dtype=torch.float32).pin_memory()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            dw = [w.to(dev, non_blocking=True) for w in wavs_host]
            host_out.copy_(expert(dw)["hidden_states"][0], non_blocking=True)
            torch.cuda.synchronize()
        e2e_ms = (time.perf_counter() - t0) * 1e3 / args.steps
    clocks = sampler.stop()
    frames = out.shape[0] * out.shape[1]
    peaks = {}
    try:
        peaks = json.loads((ROOT / "MEASURED_PEAKS.json").read_text())
    except Exception:
        pass
    peak = peaks.get("hbm_gbs", 6500.0)
    alg_bytes = sum(w.numel() * 4 for w in wavs) + out.numel() * 4
    gbs = alg_bytes / (ms_step * 1e-3) / 1e9
    line = {
        "metric": metric_name(args.config), "value": frames / (ms_step * 1e-3), "unit": "frames/s", "n_gpus": 1,
        "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(args.config, 1), "frames_per_step": frames,
                   "l2": "a 256 MB buffer is rewritten between timed iterations (L2 flush)"},
        "roofline": {"kernel": "fbank_* (warp-per-frame FFT + mel + deltas + CMVN)", "bound": "hbm", "achieved": gbs,
                     "peak": peak, "unit": "GB/s", "frac": gbs / peak, "traffic": None,
                     "note": "algorithmic bytes = waveforms in + features out (0.63 MB): the config is launch-latency bound"},
        "e2e": {"value": frames / (e2e_ms * 1e-3), "unit": "frames/s", "h2d_bytes_per_step": sum(w.numel() * 4 for w in wavs),
                "d2h_bytes_per_step": out.numel() * 4},
        "gpu_launches": 5 * args.steps,
        "clocks": clocks,
    }
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"features": out})
    if not args.no_cpu_baseline:
        fps, ms, cores, kind, timed = cpu_arm(args.config, c["batch"], 20, 2)
        line["cpu_baseline"] = {"value": fps, "unit": "frames/s", "cores": cores, "kind": kind,
                                "sample": f"the whole config (4 x 1 s), {timed} timed calls"}
    print(json.dumps(line), flush=True)


def run_ours(args):
    import torch
    import torch.distributed as dist

    from s3prl_b200 import lib as s3lib
    from s3prl_b200.upstream.expert import UpstreamExpert
    from s3prl_b200.upstream.featurizer import weighted_sum

    c = CONFIGS[args.config]
    MODEL, GLOBAL_BATCH, SECONDS = c["model"], c["batch"], c["seconds"]
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch N>1 with torch.distributed.run (one rank per GPU); see module docstring")
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=device)

    L = SECONDS * SAMPLE_RATE
    assert GLOBAL_BATCH % world == 0
    per = GLOBAL_BATCH // world
    if args.emulate_world:  # development aid: ONE rank's shard of an N-GPU run on a single GPU, no gather
        assert world == 1
        per = GLOBAL_BATCH // args.emulate_world
        GLOBAL_BATCH = per
    my_ids = list(range(rank * per, (rank + 1) * per))
    expert = UpstreamExpert(name=MODEL, seed=0).to(device)
    expert.global_max_len = L  # padding / GroupNorm statistics identical to the un-sharded batch
    if args.lanes is not None:
        expert.lanes = args.lanes
    cfg = expert.arch
    wavs_host = [seeded_wav(i, L).pin_memory() for i in my_ids]
    wavs = [w.to(device) for w in wavs_host]
    NLp1, D = cfg.encoder_layers + 1, cfg.encoder_embed_dim
    fw = torch.softmax(torch.zeros(NLp1, device=device), -1)
    T = expert.num_frames(L)
    gatherer = None
    if world > 1:
        from s3prl_b200.parallel import FeatureGatherer

        gatherer = FeatureGatherer((per, T, D), device, mode=args.gather)

    def step():
        """What a caller of the hot path receives: (hidden states, weighted-sum features)."""
        hs = expert(wavs)["hidden_states"]
        if gatherer is not None:  # weighted sum written straight into every rank's gathered buffer (or NCCL)
            return hs, gatherer.weighted_sum_gather(hs, fw)
        return hs, weighted_sum(hs, fw)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    with torch.no_grad():
        sampler = ClockSampler(local_rank) if rank == 0 else None
        if sampler:
            sampler.start()  # nvidia-smi needs ~100 ms to come up: start it before the warm-up
        # the warm-up keeps the previous step's outputs alive as the timed loop does, so that the allocator already
        # holds both output buffers when timing starts
        for _ in range(max(args.warmup, 3)):
            last = step()
        if gatherer is not None:
            gatherer.finish()
        # ---- timed region: device-resident inputs ----------------------------------------------------------
        native = expert._native
        launches0 = native.lib.s3b_launch_count(native.handle)
        barrier()
        if sampler:
            sampler.mark_begin()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        t_host = time.perf_counter()
        for _ in range(args.steps):
            last = step()
        if gatherer is not None:
            gatherer.finish()  # every rank's last gathered buffer is complete (all peers' pushes have landed)
        host_enqueue_ms = (time.perf_counter() - t_host) * 1e3 / args.steps  # CPU time to enqueue one step
        e1.record()
        barrier()
        ms_total = torch.tensor([e0.elapsed_time(e1)], device=device)
        if world > 1:
            dist.all_reduce(ms_total, op=dist.ReduceOp.MAX)
        ms_step = ms_total.item() / args.steps
        launches = (native.lib.s3b_launch_count(native.handle) - launches0) + args.steps  # + weighted-sum kernel
        frames_step = GLOBAL_BATCH * T
        value = frames_step / (ms_step * 1e-3)

        # ---- profiled pass: CUDA events around every launch, same steps (GEMM roofline) ------------------------
        import ctypes as C

        s3lib.check(native.lib.s3b_profile_enable(native.handle, 1))
        barrier()
        for _ in range(args.steps):
            step()
        if gatherer is not None:
            gatherer.finish()
        ms5, fl5, ln5 = (C.c_double * 5)(), (C.c_double * 5)(), (C.c_int64 * 5)()
        s3lib.check(native.lib.s3b_profile_read(native.handle, ms5, fl5, ln5, 1))
        s3lib.check(native.lib.s3b_profile_enable(native.handle, 0))
        clocks = sampler.stop() if sampler else None  # samples of the timed + profiled passes (same kernels, same load)
        cat = ["gemm_tcgen05", "attention_tcgen05", "conv0_norm_gelu", "layernorm", "misc"]
        breakdown = {c_: {"ms_per_step": ms5[i] / args.steps, "launches_per_step": ln5[i] // args.steps,
                          "alg_tflop_per_step": fl5[i] / args.steps / 1e12} for i, c_ in enumerate(cat)}
        gemm_tflops = (fl5[0] / 1e12) / (ms5[0] * 1e-3) if ms5[0] > 0 else 0.0

        # ---- e2e: the same step from HOST buffers -----------------------------------------------------------------
        # pinned host waveforms -> s3b_forward_host_ex (H2D, forward, every hidden state copied back to pinned host
        # memory while the next layer runs) -> weighted sum on the device-resident copy -> all-gather (N > 1) -> the
        # gathered features copied to pinned host memory. Wall clock, max over ranks.
        feat_host = torch.empty((GLOBAL_BATCH, T, D), dtype=torch.float32).pin_memory()

        e2e_gathered = torch.empty((GLOBAL_BATCH, T, D), dtype=torch.float32, device=device) if world > 1 else None

        def e2e_step():
            out_host, hs_dev = expert.forward_host(wavs_host, keep_device=True)
            feat = weighted_sum([hs_dev[i] for i in range(NLp1)], fw)
            if world > 1:
                # the end-to-end step is bound by the host<->device copies and synchronises every step anyway: plain
                # NCCL here (measured at N = 8: 3.74 M frames/s vs 2.42 M with the flag-polling push path, r2j)
                dist.all_gather_into_tensor(e2e_gathered, feat)
                feat = e2e_gathered
            feat_host.copy_(feat, non_blocking=True)
            torch.cuda.synchronize()
            return out_host

        for _ in range(2):
            e2e_step()
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            out_host = e2e_step()
        torch.cuda.synchronize()
        dt = torch.tensor([time.perf_counter() - t0], device=device)
        if world > 1:
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        e2e_value = frames_step * args.steps / dt.item()
        h2d = sum(w.numel() * 4 for w in wavs_host)
        d2h = out_host.numel() * 4

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    if args.dump_outputs:  # rank 0: the gathered features of the whole batch, the hidden states of its own shard
        hidden_states, features = last
        dump_outputs(args.dump_outputs, {"features": features, "hidden_states": hidden_states})

    peaks = {}
    try:
        peaks = json.loads((ROOT / "MEASURED_PEAKS.json").read_text())
    except Exception:
        pass
    peak_tf = peaks.get("bf16_tflops_sustained", 1400.0)
    peak_src = "MEASURED_PEAKS.json bf16_tflops_sustained (measured)" if peaks else "fallback 1.4 PFLOP/s sustained (B200_PROFILING.md)"
    flops_utt, _ = algorithmic_flops_per_utt(cfg, L)
    if args.lanes is None:  # the library's choice for this shard (two lanes from a measured frame count on)
        from s3prl_b200 import lib as _s3b_lib

        lanes_used = int(_s3b_lib.load().s3b_default_lanes(None, len(my_ids), L))
    else:
        lanes_used = args.lanes
    scheme = os.environ.get("S3B_GEMM_SCHEME", "f16q8")  # the library's default (model.cu S3B_DEFAULT_SCHEME)
    if scheme in ("1", "f16q8"):
        scheme, slots = "f16q8", 2.0
        dtype = "f32 (fp16 product + two e4m3 correction products = 2 MMA slots per 16 of K, fp32 TMEM accumulate)"
    else:
        scheme, slots = "bf16x3", 3.0
        dtype = "f32 (bf16 hi+lo split operands x3 MMAs, fp32 TMEM accumulate)"
    line = {
        "metric": metric_name(args.config), "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": dtype, "data": "synthetic",
        "config": {
            "workload": workload_name(args.config, world),
            "operand_scheme": scheme,
            "frames_per_step": frames_step,
            "l2": "activations and outputs (>= 0.64 GB of hidden states per step) exceed the 126 MB L2",
            "alg_tflop_per_step": flops_utt * GLOBAL_BATCH / 1e12,
            "lanes": lanes_used,
            "emulated_shard_of": args.emulate_world or None,
            "gather": (gatherer.mode if gatherer is not None else None),
        },
        "whole_step_tflops": flops_utt * GLOBAL_BATCH / 1e12 / (ms_step * 1e-3),
        "roofline": {
            "kernel": "gemm2_kernel (tcgen05 cta_group::2, all GEMM launches of a step)", "bound": "tensor",
            "achieved": gemm_tflops, "peak": peak_tf, "unit": "TFLOP/s", "frac": gemm_tflops / peak_tf,
            "traffic": gemm_traffic(), "peak_source": peak_src,
            "mma_pipe_tflops": slots * gemm_tflops,
            "note": "achieved = algorithmic FLOPs (1 MMA per product; the tensor pipe spends `slots` bf16-rate MMA slots per product: 3 for bf16x3, 2 for f16q8 = mma_pipe_tflops; pos_conv always runs bf16x3) / CUDA-event time per launch in a profiled pass of the same steps (lanes run one after the other there so that every kernel is timed alone at its production shape), rank 0; traffic = bytes per launch (ncu, profiles/)",
        },
        "kernel_breakdown": breakdown,
        "e2e": {"value": e2e_value, "unit": "frames/s", "h2d_bytes_per_step": h2d * world,
                "d2h_bytes_per_step": d2h * world + feat_host.numel() * 4 * world,
                "host_chunks": int(os.environ.get("S3B_HOST_CHUNKS", 2 if GLOBAL_BATCH // world >= 16 else 1)),
                "region": "H2D waveforms, forward, D2H of all hidden states (overlapped per layer), weighted sum, all-gather (N>1), D2H of the gathered features"},
        "gpu_launches": int(launches),
        "host_enqueue_ms_per_step": host_enqueue_ms,
        "clocks": clocks,
    }
    if world == 1 and not args.no_cpu_baseline:
        n_utts = 4 if SECONDS <= 10 else 2
        fps, ms, cores, kind, timed = cpu_arm(args.config, n_utts, 3, 1, budget_s=40.0)
        line["cpu_baseline"] = {"value": fps, "unit": "frames/s", "cores": cores, "kind": kind,
                                "sample": f"{n_utts} of the {GLOBAL_BATCH} utterances (x {SECONDS} s), 1 warm-up + {timed} timed passes of "
                                          + ("the reference itself (s3prl UpstreamExpert + Featurizer)" if kind == "reference" else "the oracle port")
                                          + "; the full-batch number is the --impl reference line"}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="c2", choices=sorted(CONFIGS))
    ap.add_argument("--lanes", type=int, default=None, help="utterance micro-batch lanes (default: library default)")
    ap.add_argument("--gather", default="auto", choices=["auto", "push", "nccl"],
                    help="N>1: fused weighted-sum + peer-memory push (default when peer access works) or one NCCL all-gather")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--emulate-world", type=int, default=0,
                    help="development aid: time one rank's shard of an N-GPU run on one GPU (no gather); not a bench line")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed to DIR/<name>.npy (float32, at most 64 MB in all)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes this project's outputs; it does not apply to --impl reference")
    if args.impl == "reference":
        run_reference(args)
    elif CONFIGS[args.config]["model"] == "fbank":
        run_fbank(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
