#!/usr/bin/env python
"""Benchmark of the FastSpeech2 mel-synthesis forward path on B200 (one process per GPU).

    python bench.py --gpus 1 --steps 10 --warmup 3                  # our arm, N=1
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W      # N ranks, NCCL
    python bench.py --impl reference --gpus 1 --steps 3 --warmup 1  # reference arm (CPU)
    python bench.py --gpus 1 --steps 10 --warmup 3 --dump-outputs DIR   # also write the last timed step's outputs

Metric (BASELINE.json): valid mel-frames/s of batched synthesis.  A "step" is one eval-mode
`FeedForwardTransformer._forward` over one synthetic LJSpeech-shaped batch: phoneme encoder,
duration predictor, LengthRegulator, pitch/energy predictors + embeddings, mel decoder, mel
linear, Postnet (teacher-forced durations so the frame count is fixed; SURVEY.md section 8d),
plus -- for N > 1 -- the single NCCL all-gather of the final mels.  Workload c2: B=64,
T=100 phonemes, L=800 frames per utterance per GPU (weak scaling: every rank owns its shard).

Precision: the default (and the headline `value` / `dtype`) is "3xf16" -- every contraction of the path, both attention
products included, error-compensated on the tensor cores: fp32-class results (parity gate max-abs 1e-4 against the fp32
reference, the reference's own precision).  The 10-bit-mantissa fast modes are measured beside it in `modes`.

`value`  : whole-job frames/s with inputs resident in HBM, CUDA-event timed, max over ranks.
`e2e`    : same through the public API with HOST (pinned) inputs: H2D of xs/ilens/olens/ds/es/ps
           and D2H of the mel batch inside the timed region, every step (both on side streams: two captured graphs
           with their own static inputs / outputs alternate, so the uploads of step i+1 and the mel copy of step i-1
           overlap step i; events order every copy against the replay that produces / consumes the buffer).
`roofline`: dominant kernel class (decoder conv-FFN w_1: k=9 conv 384->1024 as a tap-GEMM),
           algorithmic FLOPs per launch / its CUDA-event duration measured by the library's
           per-kernel-class event profiler on extra steps of this same workload.
`cpu_baseline`: the UNMODIFIED reference (`baseline/_ref`, staged by tools/make_baseline_ref.py) on a
           bounded sample of the same workload on the host cores (kind "reference"); the oracle port if the
           staged reference is absent (kind "port").
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

WORKLOADS = {
    # name: (B per GPU, T, L)
    "c2": (64, 100, 800),     # BASELINE.json configs[1]: batch=64 LJSpeech-length on 1xB200 (headline)
    "c4": (32, 250, 2000),    # configs[3]: long-form
    "c5": (256, 100, 0),      # configs[4]: LengthRegulator stress (ds ~ U{1..15}, alpha = 4): LR kernels only
}
HOP, SR = 256, 22050


def mflop_per_frame(T: int, L: int) -> float:
    """Algorithmic MFLOP (2*MAC) per valid mel frame, SURVEY.md section 8d table."""
    fpp = L / T
    enc = 4 * (4 * 256 ** 2 + 2 * T * 256 + 256 * 1024 * 9 + 1024 * 256) + 2 * 256 ** 2 * 3 + 256
    var = 2 * (2 * 256 ** 2 * 3 + 256)
    dec = 256 * 384 + 4 * (4 * 384 ** 2 + 2 * L * 384 + 384 * 1024 * 9 + 1024 * 384) + 384 * 80
    post = 80 * 256 * 5 + 3 * 256 ** 2 * 5 + 256 * 80 * 5
    return 2.0 * (enc / fpp + var + dec + post) / 1e6


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx, self.proc, self.lines = gpu_index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "25",
                                          "-i", str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def wait_first(self, timeout=5.0):
        t0 = time.time()
        while self.proc and not self.lines and time.time() - t0 < timeout:
            time.sleep(0.05)

    def mark(self):
        return time.time()

    def stop(self, t_begin=0.0, t_end=1e300):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for ts, ln in self.lines:
            if ts < t_begin or ts > t_end + 0.15:
                continue
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx = float(f[2])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "samples": len(sm), "reasons": sorted(reasons)}

    def median_between(self, t_begin, t_end):
        """Median SM clock of the samples inside [t_begin, t_end] (per timed loop), or None."""
        sm = []
        for ts, ln in self.lines:
            if t_begin <= ts <= t_end + 0.03:
                f = [x.strip() for x in ln.split(",")]
                try:
                    sm.append(float(f[1]))
                except (ValueError, IndexError):
                    pass
        sm.sort()
        return sm[len(sm) // 2] if sm else None


def ncu_traffic(kernel: str, precision: str = "tf32", info: bool = False):
    """DRAM bytes per launch of `kernel` in `precision` mode from the committed `ncu --set full` capture
    (profiles/ncu_traffic.json; keys are "<class>" for tf32 captures and "<class>@<precision>" otherwise), or None.
    The number is a property of the build that was captured, not of this run: `info=True` returns where it came from."""
    p = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    try:
        d = json.load(open(p))
        e = d.get(kernel if precision == "tf32" else f"{kernel}@{precision}", {})
        if info:
            return (f"{e.get('source')} ({e.get('build')})" if e else None)
        return e.get("dram_bytes_per_launch")
    except Exception:
        return None


FMA_PEAK = 2 * 148 * 128 * 1.965e9 / 1e12      # fp32 FMA pipe: 148 SM x 128 lanes x 2 flop x 1.965 GHz (nominal)


def class_peak(precision: str, cls: str, tf_peak: float):
    """Tensor / FMA peak (TFLOP/s) that bounds profiler class `cls` in `precision` mode, and how it was derived
    (DESIGN.md section 2: which instruction kind each class runs on).  `tf_peak` is the measured dense bf16 rate."""
    fma = (FMA_PEAK, "fp32 FMA pipe = 148 SM x 128 lanes x 2 x 1.965 GHz (nominal)")
    f16 = (tf_peak, "kind::f16 dense = the measured bf16 rate")
    tf32 = (tf_peak / 2.0, "kind::tf32 dense = 1/2 of the measured bf16 rate")
    x3 = (tf_peak / 3.0, "3xF16 (three kind::f16 products per term) = 1/3 of the measured bf16 rate")
    if precision == "fp32":
        return fma
    if cls.startswith("enc.") or cls.startswith("predictor.") or precision in ("3xtf32", "3xf16"):
        return x3
    return f16 if precision == "f16" else tf32


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d["hbm_gbs"], d["bf16_tflops"], d["bf16_tflops_sustained"], "measured (MEASURED_PEAKS.json)"
    return 6650.0, 1590.0, 1400.0, "fallback (B200_PROFILING.md)"


def cpu_frames_per_s(B: int, T: int, L: int, steps: int, warmup: int, threads: int = 32):
    """The reference's own CPU path on B utterances of the workload: the UNMODIFIED `FeedForwardTransformer._forward` from
    `baseline/_ref` (kind "reference"), or the oracle port when the staged reference is absent (kind "port").  PyTorch's
    CPU kernels do not scale to every core of a 128-thread host on these shapes (oversubscription makes them slower;
    measured in round 1: 16-32 threads is the optimum), so the thread count is fixed at min(32, cores) and reported."""
    from fastspeech2_b200 import synthetic_state_dict
    from fastspeech2_b200.synthetic import make_batch
    from oracle import ref_import
    cores = min(threads, os.cpu_count() or 1)
    torch.set_num_threads(cores)
    sd = synthetic_state_dict(0)
    bt = make_batch(B, T, L, seed=1234)
    if ref_import.available():
        cls, hp = ref_import.load_reference()
        model = cls(68, 80, hp)
        model.load_state_dict(sd, strict=True)
        model.eval()
        kind = "reference"

        def fwd():
            return model._forward(bt["xs"], bt["ilens"], bt["olens"], bt["ds"].clone(), bt["es"], bt["ps"], is_inference=False)
    else:
        from oracle import fs2_oracle as O
        kind = "port"

        def fwd():
            return O.forward_path(sd, bt["xs"], bt["ilens"], bt["olens"], bt["ds"].clone(), bt["es"], bt["ps"], False)
    times = []
    with torch.no_grad():
        for i in range(warmup + steps):
            t0 = time.perf_counter()
            out = fwd()
            if i >= warmup:
                times.append(time.perf_counter() - t0)
    dt = sum(times) / len(times)
    return B * L / dt, dt, cores, kind, out


DUMP_BUDGET = 60 * 10 ** 6   # bytes of array data written by --dump-outputs: under 64 MB with the .npy headers


def dump_outputs(directory: str, arrays) -> None:
    """Write {name: tensor} as DIR/<name>.npy (floating point as float32, integers as float64, both exact).  When the
    arrays exceed DUMP_BUDGET, each keeps the same share of its entries at positions drawn from a fixed seed, written
    flattened beside DIR/<name>_index.npy; the inputs of a run are seeded, so two builds can be compared file by file."""
    import numpy as np
    host = {k: v.detach().to("cpu", torch.float64 if not v.is_floating_point() or v.dtype == torch.float64 else torch.float32)
            for k, v in arrays.items()}
    total = sum(v.numel() * v.element_size() for v in host.values())
    os.makedirs(directory, exist_ok=True)
    for name, v in host.items():
        if total > DUMP_BUDGET:
            keep = max(1, int(v.numel() * (DUMP_BUDGET / 3) / total))    # float64 indices: at most twice the values' bytes
            idx = torch.randperm(v.numel(), generator=torch.Generator().manual_seed(0))[:keep].sort().values
            np.save(os.path.join(directory, f"{name}_index.npy"), idx.to(torch.float64).numpy())
            v = v.reshape(-1)[idx]
        np.save(os.path.join(directory, f"{name}.npy"), v.numpy())


def run_reference(args):
    """Reference arm: the reference's own CPU implementation of the path -- the unmodified reference class staged in
    baseline/_ref (falls back to the oracle port, which issues the same ATen calls and is pinned bit-exact to it by
    tests/golden).  Rank 0 only."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    B, T, L = WORKLOADS[args.workload]
    Bs = min(B, args.cpu_sample_batch)
    fps, dt, cores, kind, out = cpu_frames_per_s(Bs, T, L, args.steps, args.warmup, args.cpu_threads)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, dict(zip(("before_outs", "after_outs", "d_outs", "e_outs", "p_outs"), out)))
    sample = f"{Bs} of the {B} utterances of workload {args.workload} (T={T}, L={L}) per step, {cores} threads"
    line = {
        "impl": "reference", "metric": "mel-frames/sec (batched inference)", "value": fps, "unit": "frames/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": args.workload, "B_per_gpu": B, "T": T, "L": L, "mode": "teacher-forced _forward, eval, no_grad",
                   "same_config": Bs == B},
        "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "rtf": (1.0 / fps) / (HOP / SR),
    }
    print(json.dumps(line), flush=True)


def run_length_regulator(args):
    """BASELINE config 5: LengthRegulator alone, B=256, T=100, C=256, ds ~ U{1..15}, alpha=4.0 (round half even)
    -> Lmax ~ 3.7k frames, ~0.97 GB written per step.  HBM-bound: report GB/s against the measured copy peak."""
    from fastspeech2_b200 import LengthRegulator, _lib
    from oracle import fs2_oracle as O
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    lib = _lib.load()
    B, T, _ = WORKLOADS["c5"]
    g = torch.Generator().manual_seed(1234)
    hs = torch.randn(B, T, 256, generator=g)
    ds = torch.randint(1, 16, (B, T), generator=g)
    il = torch.full((B,), T, dtype=torch.int64)
    hs_d, ds_d, il_d = hs.to(dev), ds.to(dev), il.to(dev)
    hs_h, ds_h = hs.pin_memory(), ds.pin_memory()
    lr = LengthRegulator()
    out = lr(hs_d, ds_d, il_d, alpha=4.0)
    Lmax = out.shape[1]
    frames = int(torch.round(ds.float() * 4.0).long().sum())
    algo_bytes = B * T * 256 * 4 + B * T * 8 + B * Lmax * 256 * 4
    out_h = torch.empty(out.shape, dtype=torch.float32).pin_memory()

    def timed(fn, steps, warmup):
        for _ in range(warmup):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / steps

    n0 = lib.fs2_kernel_launches()
    last_out = [None]

    def step():
        last_out[0] = lr(hs_d, ds_d, il_d, alpha=4.0)
    ms = timed(step, args.steps, max(args.warmup, 3))
    launches = (lib.fs2_kernel_launches() - n0) // (args.steps + max(args.warmup, 3))
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"out": last_out[0]})

    def e2e():
        o = lr(hs_h.to(dev, non_blocking=True), ds_h.to(dev, non_blocking=True), il_d, alpha=4.0)
        out_h.copy_(o, non_blocking=True)
    ms_e2e = timed(e2e, max(2, args.steps // 2), 1)
    # the gather kernel alone (the plan kernel + the host read of Lmax are latency, not bandwidth)
    from fastspeech2_b200 import length_regulator as _lrmod
    cum, _, _, il_dev = _lrmod.plan(hs_d, ds_d, il_d, 4.0)
    ms_gather = timed(lambda: _lrmod.gather(hs_d, cum, il_dev, Lmax), args.steps, 3)
    hbm, _, _, src = peaks()
    t0 = time.perf_counter(); ref = O.length_regulator(hs, ds.clone(), il, alpha=4.0); cpu_s = time.perf_counter() - t0
    assert torch.equal(out.cpu(), ref), "LengthRegulator output differs from the oracle"
    line = {
        "metric": "mel-frames/sec (LengthRegulator only)", "value": frames / (ms * 1e-3), "unit": "frames/s", "n_gpus": 1,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32 copy / i64 scan", "data": "synthetic",
        "config": {"workload": "c5", "B": B, "T": T, "C": 256, "alpha": 4.0, "Lmax": Lmax, "bit_exact_vs_oracle": True,
                   "l2": "0.97 GB output per step >> 126 MB L2; the 26 MB input is legitimately L2-resident (each row is read ~32x)"},
        "e2e": {"value": frames / (ms_e2e * 1e-3), "unit": "frames/s", "ms_per_step": ms_e2e,
                "h2d_bytes_per_step": hs_h.numel() * 4 + ds_h.numel() * 8, "d2h_bytes_per_step": out_h.numel() * 4},
        "gpu_launches": int(launches * args.steps), "gpu_launches_per_step": int(launches),
        "roofline": {"kernel": "length_gather_kernel", "bound": "hbm", "achieved": algo_bytes / (ms_gather * 1e-3) / 1e9, "peak": hbm,
                     "unit": "GB/s", "frac": algo_bytes / (ms_gather * 1e-3) / 1e9 / hbm, "traffic": ncu_traffic("length_gather_kernel"),
                     "avg_launch_ms": ms_gather, "algorithmic_bytes": algo_bytes, "peak_source": src,
                     "whole_op_gbs": algo_bytes / (ms * 1e-3) / 1e9},
        "cpu_baseline": {"value": frames / cpu_s, "unit": "frames/s", "cores": torch.get_num_threads(), "kind": "port",
                         "sample": "one full-size call of the oracle (repeat_interleave per utterance; the reference's per-phoneme Python loop took 12.4 s in the survey)"},
    }
    print(json.dumps(line), flush=True)


def run_b200(args):
    if args.workload == "c5":
        return run_length_regulator(args)
    import torch.distributed as dist
    from fastspeech2_b200 import FeedForwardTransformer, _lib, synthetic_state_dict
    from fastspeech2_b200.hparams import load_hp
    from fastspeech2_b200.synthetic import make_batch
    from fastspeech2_b200.sharded import PeerGather, gather_mels_to_root

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torch.distributed.run --nproc-per-node {args.gpus}")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    lib = _lib.load()

    B, T, L = WORKLOADS[args.workload]
    sd = synthetic_state_dict(0)
    bt = make_batch(B, T, L, seed=1234 + rank)          # rank r owns utterances [r*B, (r+1)*B) (SURVEY.md 8e)
    keys = ("xs", "ilens", "olens", "ds", "es", "ps")
    # e2e host side = the repo's input pipeline (fastspeech2_b200/data.py): the batch is collated from per-utterance items into
    # PinnedCollator's page-locked slots (the reference's collate_tts contract), uploads are asynchronous from there
    from fastspeech2_b200.data import PinnedCollator
    items = [(bt["xs"][b, : int(bt["ilens"][b])].numpy(), bt["ys"][b, : int(bt["olens"][b])].numpy(), f"utt{b}", int(bt["olens"][b]),
              bt["ds"][b, : int(bt["ilens"][b])].numpy(), bt["es"][b, : int(bt["olens"][b])].numpy(), bt["ps"][b, : int(bt["olens"][b])].numpy())
             for b in range(B)]
    collator = PinnedCollator(B, T, L, n_mels=80, slots=2)
    pinned = [collator(items), collator(items)]                       # 9-tuples: inputs, ilens, mels, labels, olens, ids, durations, energys, pitches
    FIELD = {"xs": 0, "ilens": 1, "olens": 4, "ds": 6, "es": 7, "ps": 8}
    host = {k: pinned[0][FIELD[k]] for k in keys}
    assert all(torch.equal(host[k], bt[k]) for k in keys), "collated batch differs from the synthetic batch"
    devin = {k: bt[k].to(dev) for k in keys}
    frames_rank = int(bt["olens"].sum())
    gathered = torch.empty((world * B, L, 80), dtype=torch.float32, device=dev) if world > 1 else None
    mel_host = [torch.empty((B, L, 80), dtype=torch.float32).pin_memory() for _ in range(2)]
    copy_stream = torch.cuda.Stream(dev)      # D2H of the results
    up_stream = torch.cuda.Stream(dev)        # H2D of the inputs

    def build(precision):
        m = FeedForwardTransformer(68, 80, load_hp(), precision=precision)
        m.load_state_dict(sd, strict=True)
        return m.to(dev).eval()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    peer, collective_note = None, None
    if world > 1 and args.collective in ("peer_copy", "peer_store"):
        try:
            peer = PeerGather((B, L, 80), dev, buffers=2)      # raises on ALL ranks if any rank cannot map the root's buffer
        except Exception as e:      # no IPC / peer access on this box: say so and use the NCCL gather instead of dying
            peer = None
            args.collective = "gather"
            collective_note = f"peer_copy unavailable ({type(e).__name__}: {str(e)[:160]}); fell back to the NCCL gather"
    step_no = [0]
    last_out = [None]           # what the last device-resident step returned (--dump-outputs)

    def timed(fn, steps, warmup):
        for i in range(warmup):
            fn(i)
        barrier()
        if args.settle_s > 0:      # both timed loops start from the same power state (the 1 kW cap is a moving average: a loop
            time.sleep(args.settle_s)   # that follows another one back to back starts with the clocks already pulled down)
            barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            fn(i)
        if peer is not None:      # the timed region ends when the last shard has landed on the root, not when it was enqueued
            if rank == 0:
                peer.wait(step_no[0])
            elif peer.pushed is not None:
                torch.cuda.current_stream(dev).wait_event(peer.pushed)
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t)
        return ms / steps

    def make_steps(model):
        """(device-resident step, end-to-end step, flush) for one model.  Graph mode: two captured graphs with their own
        static inputs / outputs alternate, so the D2H copy of step i (side stream) overlaps step i+1; the length
        validation is deferred (checked at the start of the next call), so replays queue back to back."""
        fused = peer is not None and args.collective == "peer_store" and args.graph
        # fused exchange: the last Postnet kernel of graph i stores its mels straight into this rank's slot of the root's
        # receive buffer i (peer-mapped over NVLink on the other ranks)
        graphs = [model.graphed_forward(*[devin[k] for k in keys], after_out=(peer.slot(i) if fused else None)) for i in range(2)] if args.graph else None
        copied = [torch.cuda.Event(), torch.cuda.Event()]
        uploaded = [torch.cuda.Event(), torch.cuda.Event()]
        consumed = [None, None]                 # graph i's static inputs may be overwritten once its last replay has finished

        pushed = [None, None]
        big_host = ([torch.empty((world * B, L, 80), dtype=torch.float32).pin_memory() for _ in range(2)]
                    if (fused and rank == 0) else None)

        def collective(mel, i):
            if world == 1:
                return
            # the single exchange step: gather the final mel batch over NVLink
            if fused:                           # the mels are already in the root's buffer: publish the step with one flag store
                step_no[0] += 1
                peer.signal(step_no[0])
            elif peer is not None:              # copy-engine push into the root's buffer on a side stream (csrc/peer.cu)
                step_no[0] += 1
                peer.push(mel, step_no[0])
                pushed[i & 1] = peer.pushed     # this graph's output buffer is busy until the transfer has read it
            elif args.collective == "none":     # diagnostic: no exchange at all (what N independent replicas cost under max-over-ranks timing)
                pass
            elif args.collective == "gather":   # NCCL: rank 0 receives everything, the others only send their shard
                gather_mels_to_root(mel, dst=0, out=gathered if rank == 0 else None)
            else:                               # NCCL all-gather: every rank receives every shard
                dist.all_gather_into_tensor(gathered, mel)

        def source_free(i):
            if pushed[i & 1] is not None:
                torch.cuda.current_stream(dev).wait_event(pushed[i & 1])

        def step(i):
            with torch.no_grad():
                if graphs is not None:
                    source_free(i)
                    out = graphs[i & 1].replay(validate="deferred")    # inputs already sit in the graph's static buffers
                else:
                    out = model._forward(*[devin[k] for k in keys], is_inference=False)
            collective(out[1], i)
            last_out[0] = out
            return out[1]

        def step_e2e(i):
            cur = torch.cuda.current_stream(dev)
            with torch.no_grad():
                if graphs is not None:
                    g = graphs[i & 1]
                    source_free(i)
                    cur.wait_event(copied[i & 1])                       # its previous output has left for the host
                    col = pinned[i & 1]
                    dst9 = [None] * 9
                    for dst, k in zip(g.inputs, keys):
                        dst9[FIELD[k]] = dst
                    # H2D from the pinned slot straight into the graph's static inputs, on the upload stream: step i's
                    # inputs travel while step i-1 computes (they only wait for this graph's previous replay, step i-2)
                    with torch.cuda.stream(up_stream):
                        if consumed[i & 1] is not None:
                            up_stream.wait_event(consumed[i & 1])
                        collator.upload_into(col, dst9)
                        uploaded[i & 1].record(up_stream)
                    cur.wait_event(uploaded[i & 1])
                    out = g.replay(validate="deferred")
                    consumed[i & 1] = torch.cuda.Event()
                    consumed[i & 1].record(cur)
                else:
                    up = collator.to_device(pinned[i & 1], dev)
                    inp = [up[FIELD[k]] for k in keys]
                    out = model._forward(*inp, is_inference=False)
            collective(out[1], i)
            src, dst = out[1], mel_host[i & 1]
            if fused:                           # the batch lives on the root only: the root reads ALL shards back, the others nothing
                if rank != 0:
                    return out[1]
                peer.wait(step_no[0])           # every rank's shard of this step has landed
                src, dst = peer.gathered_buffer(i & 1), big_host[i & 1]
            done = torch.cuda.Event()
            done.record(cur)
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(done)
                dst.copy_(src, non_blocking=True)
                copied[i & 1].record(copy_stream)
            return out[1]

        def flush():
            if graphs is not None:
                for g in graphs:
                    g.flush()
            copy_stream.synchronize()
            up_stream.synchronize()
        return step, step_e2e, flush

    model = build(args.precision)
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
        sampler.wait_first()
    with torch.no_grad():   # count the library's launches on a warm eager step (a graph replay issues the same kernels)
        model._forward(*[devin[k] for k in keys], is_inference=False)   # first call also packs the weights: not counted
        n0 = lib.fs2_kernel_launches()
        model._forward(*[devin[k] for k in keys], is_inference=False)
    launches_per_step = lib.fs2_kernel_launches() - n0
    step, step_e2e, flush = make_steps(model)
    for i in range(max(args.warmup, 3)):
        step(i)
    torch.cuda.synchronize()
    t_begin = time.time()
    outputs = None

    def keep_outputs():         # the last timed step's (before_outs, after_outs, d_outs, e_outs, p_outs), on the host
        nonlocal outputs
        if args.dump_outputs and rank == 0:
            names = ("before_outs", "after_outs", "d_outs", "e_outs", "p_outs")
            outputs = {n: t.to("cpu") for n, t in zip(names, last_out[0])}

    if args.e2e_first:                      # diagnostic: does the e2e - value gap follow the loop order (clock sag under the power cap)?
        ms_e2e = timed(step_e2e, args.steps, 2); flush()
        t_mid = time.time()
        ms_step = timed(step, args.steps, 0); flush(); keep_outputs()
    else:
        ms_step = timed(step, args.steps, 0); flush(); keep_outputs()
        t_mid = time.time()
        ms_e2e = timed(step_e2e, args.steps, 2); flush()
    t_end = time.time()
    clocks = sampler.stop(t_begin, t_end) if sampler else None
    if clocks is not None:
        first, second = sampler.median_between(t_begin, t_mid), sampler.median_between(t_mid, t_end)
        clocks["sm_mhz_value_loop"], clocks["sm_mhz_e2e_loop"] = (second, first) if args.e2e_first else (first, second)
        clocks["window"] = f"samples every 25 ms over the device-timed loop and the e2e loop; {args.settle_s} s idle before each timed loop so both start from the same power-cap state"

    # per-kernel-class CUDA-event profile on extra steps of the same workload
    prof = None
    if rank == 0 and hasattr(lib, "fs2_profile_enable"):
        import ctypes as C
        h = model._handle
        lib.fs2_profile_enable(h, 1)
        for _ in range(3):   # local forward only: the other ranks are not in this loop, so no collective here
            with torch.no_grad():
                model._forward(devin["xs"], devin["ilens"], devin["olens"], devin["ds"], devin["es"], devin["ps"], is_inference=False)
        torch.cuda.synchronize()
        n = lib.fs2_profile_classes()
        ms = (C.c_double * n)(); cnt = (C.c_int64 * n)(); fl = (C.c_double * n)(); by = (C.c_double * n)()
        lib.fs2_profile_read(h, ms, cnt, fl, by)
        lib.fs2_profile_enable(h, 0)
        prof = {lib.fs2_profile_label(i).decode(): {"ms": ms[i], "launches": cnt[i], "flop": fl[i], "bytes": by[i]}
                for i in range(n) if cnt[i]}

    # secondary figure: the literal inference mode (predicted durations, unmasked decoder, one host read of Lmax)
    inf = None
    if rank == 0 and args.gpus == 1:
        with torch.no_grad():
            out = model._forward(devin["xs"], devin["ilens"], is_inference=True, _one_hot=False)
            inf_frames = int(out[2].sum())
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize(); e0.record()
            for _ in range(5):
                model._forward(devin["xs"], devin["ilens"], is_inference=True, _one_hot=False)
            e1.record(); torch.cuda.synchronize()
        inf = {"value": inf_frames / (e0.elapsed_time(e1) / 5 * 1e-3), "unit": "frames/s", "ms_per_step": e0.elapsed_time(e1) / 5,
               "frames_per_batch": inf_frames, "Lmax": int(out[1].shape[1]),
               "note": "is_inference=True: durations predicted on the device, decoder unmasked over the [B,Lmax] rectangle, eager launches"}

    # serving latency of one ~50-phoneme utterance through model.inference (BASELINE config 1 shape; eager launches,
    # one host read of the predicted length)
    lat = None
    if rank == 0 and args.gpus == 1:
        x1 = make_batch(1, 50, 400, seed=7)["xs"][0].to(dev)
        with torch.no_grad():
            for _ in range(3):
                mel1 = model.inference(x1)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(20):
                mel1 = model.inference(x1)
            torch.cuda.synchronize()
        lat_ms = (time.perf_counter() - t0) / 20 * 1e3
        lat = {"ms": lat_ms, "frames": int(mel1.shape[0]), "rtf": (lat_ms * 1e-3) / (mel1.shape[0] * HOP / SR),
               "note": "model.inference(x) for one 50-phoneme utterance, wall clock incl. the host read of Lmax"}

    # the 10-bit-mantissa fast modes beside the headline (same workload, same timing rules; N = 1 only)
    modes = None
    if world == 1 and args.modes:
        modes = {}
        del step, step_e2e, flush
        for prec in [p_ for p_ in args.modes.split(",") if p_ and p_ != args.precision]:
            m2 = build(prec)
            st2, st2_e2e, fl2 = make_steps(m2)
            for i in range(3):
                st2(i)
            torch.cuda.synchronize()
            ms2 = timed(st2, args.steps, 0); fl2()
            ms2e = timed(st2_e2e, args.steps, 2); fl2()
            modes[prec] = {"value": frames_rank / (ms2 * 1e-3), "unit": "frames/s", "ms_per_step": ms2,
                           "e2e": frames_rank / (ms2e * 1e-3), "e2e_ms_per_step": ms2e,
                           "tolerance": {"f16": "max-abs 5e-3, mean-abs 5e-4", "tf32": "max-abs 1e-2, mean-abs 1e-3",
                                         "fp32": "max-abs 1e-4"}.get(prec, "max-abs 1e-4, mean-abs 1e-5") + " vs the fp32 reference"}
            del m2, st2, st2_e2e, fl2
            torch.cuda.empty_cache()

    if peer is not None:
        peer.close()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    if outputs is not None:
        dump_outputs(args.dump_outputs, outputs)

    hbm, tf_burst, tf_sus, peak_src = peaks()
    frames = frames_rank * world
    value = frames / (ms_step * 1e-3)
    e2e = frames / (ms_e2e * 1e-3)
    h2d = sum(host[k].numel() * host[k].element_size() for k in keys)
    d2h = mel_host[0].numel() * 4 * (world if (peer is not None and args.collective == "peer_store" and args.graph) else 1)
    mf = mflop_per_frame(T, L)
    roof = None
    gpu_busy = None
    if prof:
        tot = sum(v["ms"] for v in prof.values())
        gpu_busy = tot / 3
        top = max(prof, key=lambda k: prof[k]["ms"])
        # a kernel class timed launch by launch with events at full clocks inside a ~10 ms step: the burst figure applies
        tensor_peak, peak_note = class_peak(args.precision, top, tf_burst)
        pk = prof[top]
        achieved = pk["flop"] / (pk["ms"] * 1e-3) / 1e12 if pk["ms"] > 0 else 0.0
        roof = {"kernel": top, "bound": "tensor", "achieved": achieved, "peak": tensor_peak, "unit": "TFLOP/s",
                "frac": achieved / tensor_peak, "traffic": ncu_traffic(top, args.precision),
                "traffic_source": ncu_traffic(top, args.precision, info=True),
                "algorithmic_bytes_per_launch": pk["bytes"] / pk["launches"], "algorithmic_flop_per_launch": pk["flop"] / pk["launches"],
                "avg_launch_ms": pk["ms"] / pk["launches"], "share_of_step": pk["ms"] / tot,
                "peak_source": peak_src + " burst bf16 figure (kernel timed alone by CUDA events); " + peak_note,
                "whole_step_frac_of_burst": (value / world * mf / 1e6) / (tf_burst / (3.0 if args.precision in ("3xtf32", "3xf16") else 1.0)),
                "classes": {k: {"ms_per_step": v["ms"] / 3, "launches_per_step": v["launches"] // 3,
                                "tflops": (v["flop"] / (v["ms"] * 1e-3) / 1e12) if v["ms"] > 0 else None,
                                "gbs": (v["bytes"] / (v["ms"] * 1e-3) / 1e9) if v["ms"] > 0 else None} for k, v in prof.items()}}
    cpu = cpu_frames_per_s(min(B, args.cpu_sample_batch), T, L, 1, 1, args.cpu_threads) if args.gpus == 1 else None
    line = {
        "metric": "mel-frames/sec (batched inference)", "value": value, "unit": "frames/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": args.precision, "data": "synthetic",
        "config": {"workload": args.workload, "B_per_gpu": B, "global_batch": B * world, "T": T, "L": L,
                   "mode": "teacher-forced _forward, eval, no_grad" + (", one CUDA graph per step" if args.graph else ", eager launches"),
                   "parallelism": f"dp{world}",
                   "precision": {"3xf16": "fp32-class: every contraction incl. attention error-compensated on tcgen05 (fp16 hi+lo operand planes, 3 products per term, fp32 accumulation)",
                                 "3xtf32": "fp32-class: every contraction incl. attention error-compensated on tcgen05 (fp16 hi+lo operand planes, 3 products per term, fp32 accumulation)",
                                 "f16": "decoder side on kind::f16 (10-bit mantissa operands), encoder + predictors error-compensated",
                                 "tf32": "decoder side on kind::tf32, encoder + predictors error-compensated",
                                 "fp32": "fp32 FMA on CUDA cores"}[args.precision],
                   "collective": ({"peer_copy": "gather to rank 0 over NVLink peer memory: one copy-engine transfer of the [B,L,80] shard per rank on a side stream + flag words (csrc/peer.cu), no SM-occupying collective kernel",
                                   "peer_store": "gather to rank 0 fused into the last Postnet kernel: its epilogue stores the [B,L,80] mels straight into the root's receive buffer over NVLink (peer-mapped output pointer) + one flag store per step; no collective kernel, no extra transfer",
                                   "gather": "one NCCL gather of the [B,L,80] mel shard to rank 0",
                                   "all_gather": "one NCCL all-gather of the [B,L,80] mel shard",
                                   "none": "DIAGNOSTIC: no exchange step (independent replicas; not a valid multi-GPU number)"}[args.collective] if world > 1 else "none"),
                   "l2": "per-step working set ~0.9 GB of activations >> 126 MB L2; no flush needed",
                   "tolerance": "3xf16 (default): max-abs 1e-4, mean-abs 1e-5 vs the CPU fp32 oracle on the mels, durations / bucket ids bit-exact; "
                                "fp32: 1e-4; f16: 5e-3 / 5e-4; tf32: 1e-2 / 1e-3 (tests/test_gpu_parity.py)"},
        "e2e": {"value": e2e, "unit": "frames/s", "ms_per_step": ms_e2e, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
        "collective_note": collective_note,
        "gpu_launches": int(launches_per_step * args.steps),
        "gpu_launches_per_step": int(launches_per_step),
        "gpu_busy_ms_per_step": gpu_busy,
        "gpu_busy_note": "sum of the per-kernel CUDA-event durations of one eager step (library profiler); value's ms_per_step is K graph replays queued back to back",
        "clocks": clocks,
        "rtf": (1.0 / value) / (HOP / SR),
        "model_tflops": value * mf / 1e6,
        "mflop_per_frame": mf,
    }
    if modes:
        line["modes"] = modes
    if inf:
        line["inference_mode"] = inf
    if lat:
        line["single_utterance_latency"] = lat
    if roof:
        line["roofline"] = roof
    if cpu:
        cpu_fps, cpu_dt, cores, kind, _ = cpu
        line["cpu_baseline"] = {"value": cpu_fps, "unit": "frames/s", "cores": cores, "kind": kind,
                                "sample": f"{min(B, args.cpu_sample_batch)} of the {B} utterances of workload {args.workload}, 1 warm-up + 1 timed forward, {cores} threads"}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS))
    ap.add_argument("--precision", default=os.environ.get("FS2_PRECISION", "3xf16"), choices=["fp32", "tf32", "3xtf32", "3xf16", "f16"])
    ap.add_argument("--modes", default="f16,tf32", help="N=1: other precision modes measured beside the headline ('' = none)")
    ap.add_argument("--cpu-sample-batch", type=int, default=64, help="utterances per CPU-reference step (64 = the full c2 batch)")
    ap.add_argument("--cpu-threads", type=int, default=32, help="host threads of the CPU reference (fixed; oversubscription is slower)")
    ap.add_argument("--collective", default="peer_store", choices=["peer_store", "peer_copy", "all_gather", "gather", "none"],
                    help="N>1 exchange step: peer_store = the last Postnet kernel stores the mels straight into rank 0's receive buffer over "
                         "NVLink (default); peer_copy = one copy-engine push per rank on a side stream; gather / all_gather = NCCL; none = diagnostic")
    ap.add_argument("--settle-s", type=float, default=0.5, help="idle seconds before every timed loop (same power-cap state for each)")
    ap.add_argument("--e2e-first", type=int, default=0, help="diagnostic: time the e2e loop before the device-resident loop")
    ap.add_argument("--graph", type=int, default=1, help="1: replay the step as one CUDA graph (default), 0: eager launches")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last device-resident timed step returned as DIR/<name>.npy "
                         "(rank 0; at most 64 MB in all, a seeded sample beyond that)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
