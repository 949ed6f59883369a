#!/usr/bin/env python
"""bench.py — speaker-embeddings/sec of the ResCNN hot path (BASELINE.json metric).

    python bench.py --gpus 1 --steps K --warmup W            # our arm, one B200
    torchrun ... bench.py --gpus N --steps K --warmup W      # N ranks, one per GPU
    python bench.py --impl reference --steps K --warmup W    # the reference's CPU path (oracle port) on host cores
    python bench.py ... --dump-outputs DIR                   # also save what the timed steps computed, DIR/<name>.npy

Headline (the JSON line's own keys): a "step" is one forward of the hot path over one batch of 64 synthetic utterances
(64 fbank x 160 frames -> 512-d), BASELINE.json configs[1]; N ranks = N utterance-sharded replicas, no collective.
Every workload runs W untimed warm-up steps, then ONE timed window of exactly K steps (CUDA events, max over ranks),
which opens once the host has queued its first steps (see hold()).
All inputs and weights come from fixed seeds, so the same arguments give the same inputs in every run, and the outputs
saved by --dump-outputs can be compared between two builds.

Sub-records of the same line (default --workload all):
  "train"    : the triplet training step of BASELINE configs[2] (N=1) / configs[4] (N=8: data parallel, ONE NCCL
               allreduce of the flat gradient bucket per step, fused Adagrad), with its own roofline and CPU baseline;
  "allpairs" : the 1024-utterance all-pairs distance + top-8 select of configs[3] (rank 0, single GPU).
One JSON line is printed by rank 0.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the benchmark leaves the source tree as it found it (it may be read-only)

METRIC = "speaker-embeddings/sec (64-fbank x 160-frame -> 512-d)"
FLOP_PER_EMB = 2306670592            # BASELINE.md §2 (forward)
CONV_TC_FLOP_PER_EMB = 2296381440    # the 11 tensor-core convs: 8 x 3x3 (94,371,840 MAC) + 3 x 5x5 s2 (131,072,000 MAC)
L2_BYTES = 126 * 1024 * 1024


_REAL_STDOUT = None


def emit(line: dict):
    """Print the single JSON result line on the real stdout."""
    sys.stdout.flush()
    if _REAL_STDOUT is not None:
        os.dup2(_REAL_STDOUT, 1)
    print(json.dumps(line), flush=True)
    if _REAL_STDOUT is not None:
        os.dup2(2, 1)   # whatever libraries print from here on (NCCL at teardown with NCCL_DEBUG=INFO) goes to stderr again


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"tflops_burst": d.get("bf16_tflops"), "tflops_sustained": d.get("bf16_tflops_sustained"),
                "hbm_gbs": d.get("hbm_gbs"), "source": "measured (MEASURED_PEAKS.json)"}
    return {"tflops_burst": 1590.0, "tflops_sustained": 1400.0, "hbm_gbs": 6650.0,
            "source": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.lines = []
        self.first = 0

    def mark(self):
        """Call at the start of the timed region: nvidia-smi needs up to a second to start, so the sampler is
        launched before warm-up and only the samples taken after this mark are reported."""
        t0 = time.time()
        while self.proc and not self.lines and time.time() - t0 < 3.0:
            time.sleep(0.01)
        self.first = len(self.lines)

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for ln in self.lines[self.first:]:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "samples": len(sm),
                "reasons": sorted(reasons)}


def make_model(dtype, device):
    """DeepSpeakerModel(512, 1211) with the reference's init and non-trivial BN statistics (SURVEY §8d)."""
    import torch

    from deepspeaker_pytorch_b200 import DeepSpeakerModel

    torch.manual_seed(0)
    m = DeepSpeakerModel(512, 1211, operand_dtype=dtype)
    g = torch.Generator().manual_seed(1)
    for mod in m.modules():
        if isinstance(mod, torch.nn.BatchNorm2d):
            mod.weight.data.uniform_(0.5, 1.5, generator=g)
            mod.bias.data.normal_(0, 0.1, generator=g)
            mod.running_mean.normal_(0, 0.1, generator=g)
            mod.running_var.uniform_(0.5, 1.5, generator=g)
    return m.to(device).eval()


def pick_cpu_threads(sd, T):
    """The reference runs on 'all the host threads it can use'; on many-core hosts oversubscribing the
    torch CPU kernels is slower than a subset, so the baseline gets the best of a few thread counts."""
    import torch

    from oracle import rescnn_oracle as O

    ncpu = os.cpu_count() or 1
    cands = sorted({c for c in (8, 16, 32, 64, ncpu) if c <= ncpu})
    x = O.make_input(16, T, seed=0)
    best, best_rate = cands[-1], 0.0
    with torch.no_grad():
        for c in cands:
            torch.set_num_threads(c)
            O.forward(sd, x)
            t0 = time.perf_counter()
            O.forward(sd, x)
            rate = 16 / (time.perf_counter() - t0)
            if rate > best_rate:
                best, best_rate = c, rate
    return best


def cpu_forward_timer(sd, B, T, budget_s, threads):
    """Times the oracle's eval forward (restatement of the reference's model.py:185-218) on host cores."""
    import torch

    from oracle import rescnn_oracle as O

    torch.set_num_threads(threads)
    x = O.make_input(B, T, seed=0)
    with torch.no_grad():
        O.forward(sd, x)  # warm-up
        t0 = time.perf_counter()
        n = 0
        while True:
            O.forward(sd, x)
            n += 1
            el = time.perf_counter() - t0
            if el > budget_s or n >= 50:
                break
    return B * n / el, n, el



def workload_config(args, world, dtype_note=True):
    """The `config` object of the JSON line: identical for our arm and the reference arm, so the two lines compare."""
    B, T = args.batch, args.frames
    in_bytes = B * T * 64 * 4
    nbuf = L2_BYTES // in_bytes + 8
    return {"workload": f"batch-{B} embedding inference, synthetic 64x{T} fbank, eval-mode BN, "
                        f"DeepSpeakerModel(512,1211) random init (BASELINE configs[1])",
            "batch_per_gpu": B, "frames": T, "parallelism": f"replicas x{world} (utterance-sharded, no collective)",
            "l2": f"inputs rotate over {nbuf} buffers = {nbuf * in_bytes >> 20} MiB > 126 MiB L2; "
                  f"activations ({B * 1843200 >> 20} MiB/step) are rewritten every step"}


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU implementation of the path, run as the oracle port (the same PyTorch
    CPU kernels the reference dispatches to), so that no copy of the reference is needed."""
    if rank != 0:
        return
    import torch

    from oracle import rescnn_oracle as O

    sd = {k: v for k, v in make_model("fp16", "cpu").state_dict().items()}
    B, T = args.batch, args.frames
    threads = pick_cpu_threads(sd, T)
    torch.set_num_threads(threads)
    x = O.make_input(B, T, seed=0)
    with torch.no_grad():
        t0 = time.perf_counter()
        O.forward(sd, x)
        t1 = time.perf_counter() - t0
        # bound the whole run to ~2 minutes: shrink the per-step sample if needed
        total = (args.steps + args.warmup) * t1
        b = B if total <= 120 else max(1, int(B * 120 / total))
        xs = x[:b]
        for _ in range(args.warmup):
            O.forward(sd, xs)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            O.forward(sd, xs)
        el = time.perf_counter() - t0
    val = b * args.steps / el
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": "emb/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": el / args.steps * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, max(1, args.gpus)),
        "cpu_baseline": {"value": val, "unit": "emb/s", "cores": threads, "host_cpus": os.cpu_count(),
                         "kind": "port",
                         "sample": f"{args.steps} steps x {b} utterances of the batch-{B} workload (oracle port of "
                                   f"model.py:185-218 on torch CPU fp32 kernels)"},
        "e2e": {"value": val, "unit": "emb/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    emit(line)


class Dist:
    """Rank / world plumbing shared by the three workloads (torch.distributed over NCCL when world > 1)."""

    def __init__(self, rank, world, local_rank):
        import torch

        self.rank, self.world, self.local_rank = rank, world, local_rank
        self.dev = torch.device("cuda", local_rank)

    def barrier(self):
        import torch
        import torch.distributed as dist

        if self.world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(self, values):
        """element-wise max over ranks of a list of floats (window times)"""
        import torch
        import torch.distributed as dist

        if self.world == 1:
            return list(values)
        t = torch.tensor(list(values), device=self.dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.tolist()


def timed_window(D, window):
    """Runs the timed window once: exactly --steps steps, bracketed by barrier + synchronize on both sides, CUDA events
    on the launching stream.  Returns its milliseconds, the max over ranks."""
    return D.max_over_ranks([window()])[0]


HOLD_CYCLES = 20_000_000    # ~10 ms at the B200's 1965 MHz boost clock


def hold(stream):
    """Called between a window's opening synchronize and its first event: keeps `stream` busy for ~10 ms (one spinning
    thread) so that the host has queued the window's first steps before they can start.  Every stream of a step orders
    after the launching stream, so the window times the steps back to back.  A 20-step inference window lasts 3.6 ms, and
    without the hold it also timed any delay of the host thread while it queued them: on a B200 (1000 W limit) single
    windows then ranged from 33 k to 353 k emb/s, with it 353.1 k to 353.7 k."""
    import torch

    with torch.cuda.stream(stream):
        torch.cuda._sleep(HOLD_CYCLES)


DUMP_MAX_ELEMS = 1 << 20    # per array (4 MB in fp32, 8 MB in fp64): the seven arrays of a run stay well below 64 MB in all


def write_outputs(out_dir, outputs):
    """--dump-outputs: one DIR/<name>.npy per array of what the timed steps computed in their last step, float32 (float64
    for integer results, which it holds exactly).  An array above DUMP_MAX_ELEMS is replaced by a fixed, seeded sample of
    its flattened elements, so two runs with the same arguments sample the same positions."""
    import numpy as np

    os.makedirs(out_dir, exist_ok=True)
    for name, a in outputs.items():
        a = np.asarray(a)
        a = a.astype(np.float32 if a.dtype.kind == "f" else np.float64)
        if a.size > DUMP_MAX_ELEMS:
            a = a.reshape(-1)[np.sort(np.random.default_rng(0).choice(a.size, DUMP_MAX_ELEMS, replace=False))]
        np.save(os.path.join(out_dir, name + ".npy"), a)


def conv_kernel_hash():
    """Content hash of the dominant kernel's sources: profiles/traffic.json stores the ncu DRAM traffic per build."""
    import hashlib

    h = hashlib.sha1()
    for f in ("conv3x3_halo.cuh", "conv_umma.cuh", "dsk_ptx.cuh"):
        with open(os.path.join(ROOT, "deepspeaker_pytorch_b200", "csrc", f), "rb") as fh:
            h.update(fh.read())
    return h.hexdigest()[:12]


def measured_traffic(B, T):
    """dram__bytes_read.sum + dram__bytes_write.sum of the 11 tensor-core conv launches of one forward, from the
    committed `ncu --set full` capture of THIS kernel build (profiles/traffic.json), else None."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            table = json.load(f)
    except (OSError, ValueError):
        return None, "profiles/traffic.json missing"
    key = conv_kernel_hash()
    for e in table.get("captures", []):
        if e.get("kernel_hash") == key and e.get("batch") == B and e.get("frames") == T:
            return e["dram_bytes_per_forward"], e.get("source")
    return None, f"no ncu capture recorded for kernel build {key} at batch {B}"


def bench_infer(args, D, outputs):
    """The headline: batch-64 eval inference (BASELINE configs[1]) through EmbeddingPipeline.  Puts the embeddings of
    the last timed step into `outputs`."""
    import ctypes

    import torch

    from deepspeaker_pytorch_b200 import EmbeddingPipeline
    from deepspeaker_pytorch_b200 import _lib as L

    dev, rank, world = D.dev, D.rank, D.world
    B, T, K, W = args.batch, args.frames, args.steps, args.warmup
    model = make_model(args.dtype, dev)
    in_bytes = B * T * 64 * 4
    nbuf = L2_BYTES // in_bytes + 8  # rotating inputs larger than L2
    g = torch.Generator(device=dev).manual_seed(rank)
    xs = [torch.randn(B, 1, T, 64, device=dev, generator=g) for _ in range(nbuf)]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    pipe = EmbeddingPipeline(model, lanes=args.lanes)
    cur = torch.cuda.current_stream(dev)
    cnt = [0]
    host_ms = []
    last = [None]
    with torch.no_grad():
        sampler = ClockSampler(D.local_rank)
        if rank == 0:
            sampler.start()
        # one-time setup outside the W warm-up steps: every lane builds its plan (first call) and captures its CUDA
        # graph (second call), so a short --steps run does not time graph instantiation
        for i in range(2 * args.lanes):
            pipe.embed_device(xs[i % nbuf])
        pipe.synchronize()
        # the clock samples start here, and the warm-up steps follow at once: no idle gap before the timed window
        D.barrier()
        if rank == 0:
            sampler.mark()
        for i in range(W):
            pipe.embed_device(xs[i % nbuf])
        pipe.synchronize()

        # ---- value: inputs resident in HBM; `lanes` forwards in flight through the public pipeline ------------------
        def window():
            D.barrier()
            hold(cur)
            e0.record(cur)
            t_host = time.perf_counter()
            for _ in range(K):
                last[0] = pipe.embed_device(xs[cnt[0] % nbuf])
                cnt[0] += 1
            host_ms.append((time.perf_counter() - t_host) * 1e3 / K)
            for st in pipe.lanes:
                cur.wait_stream(st)
            e1.record(cur)
            D.barrier()
            return e0.elapsed_time(e1)

        ms = timed_window(D, window)
        value = world * B * K / (ms * 1e-3)
        host_ms_value = host_ms[0]
        outputs["embeddings"] = last[0].cpu().numpy()

        # ---- e2e: host buffers through the public API, H2D + D2H inside the timed region -----------
        nhost = 8
        xh = [torch.randn(B, 1, T, 64).pin_memory() for _ in range(nhost)]
        oh = [torch.empty(B, 512).pin_memory() for _ in range(nhost)]
        # one-time setup outside the W warm-up steps: the pipeline allocates the device buffers of each of its
        # lanes x depth staging slots at the slot's first use, so every slot is used once before the timed window
        for i in range(len(pipe.lanes) * pipe.depth):
            pipe.embed(xh[i % nhost], oh[i % nhost])
        pipe.synchronize()
        for i in range(W):
            pipe.embed(xh[i % nhost], oh[i % nhost])
        pipe.synchronize()
        host_ms2 = []

        def window_e2e():
            D.barrier()
            hold(pipe.h2d)
            e0.record(pipe.h2d)
            t_host = time.perf_counter()
            for _ in range(K):
                pipe.embed(xh[cnt[0] % nhost], oh[cnt[0] % nhost])
                cnt[0] += 1
            host_ms2.append((time.perf_counter() - t_host) * 1e3 / K)
            e1.record(pipe.d2h)     # the D2H stream is in order: this event follows the last batch's copy-out
            pipe.synchronize()
            D.barrier()
            return e0.elapsed_time(e1)

        ms_e2e = timed_window(D, window_e2e)
        clocks = sampler.stop() if rank == 0 else None
        e2e_value = world * B * K / (ms_e2e * 1e-3)
        host_ms_e2e = host_ms2[0]

        # ---- roofline of the dominant kernel: per-launch CUDA-event times inside the forward ---------
        eng = model._engine
        buf = (ctypes.c_float * 32)()
        n = ctypes.c_int32(0)
        nprof = 20

        def profile(level):
            L.check(eng.lib.dsk_set_profiling(eng.handle, level))
            acc = None
            for i in range(nprof):
                model(xs[i % nbuf])
                L.check(eng.lib.dsk_get_launch_times(eng.handle, buf, 32, ctypes.byref(n)))
                v = [buf[j] for j in range(n.value)]
                acc = v if acc is None else [a + b for a, b in zip(acc, v)]
            L.check(eng.lib.dsk_set_profiling(eng.handle, 0))
            return [a / nprof for a in acc]

        # level 2: events only at the section boundaries conv1 | 11 tensor-core convs | tail, so the conv launches run
        # back to back as in production; level 1: an event after every launch (adds ~5 us of event latency to each)
        sec_ms = profile(2)
        per_launch_ms = profile(1)
    if rank != 0:
        return None
    conv_ms = sec_ms[1]
    step_ms_prof = sum(sec_ms)
    peaks = load_peaks()
    achieved = B * CONV_TC_FLOP_PER_EMB / (conv_ms * 1e-3) / 1e12
    # the conv chain is timed alone (one forward, two events): the burst figure of MEASURED_PEAKS is its denominator; the
    # sustained figure belongs to the in-production rate, which is measured inside a long back-to-back run
    peak = peaks["tflops_burst"]
    traffic, traffic_src = measured_traffic(B, T)
    # the production step keeps `lanes` forwards in flight, so launches of different forwards overlap: the in-production
    # rate charges the conv FLOPs with the WHOLE measured step (conv1 and the tail run under other forwards' convs)
    share = conv_ms / step_ms_prof
    overlapped = B * CONV_TC_FLOP_PER_EMB / (ms / K * 1e-3) / 1e12
    roofline = {
        "bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
        "traffic": traffic, "traffic_source": traffic_src,
        "kernel": "conv3x3_halo_kernel: the 11 tensor-core conv launches of a step (8 x 3x3 s1 + 3 x parity-planar 5x5 s2), "
                  "timed back to back between two CUDA events on the forward's stream (one forward in flight)",
        "flop_per_launch_set": B * CONV_TC_FLOP_PER_EMB, "launch_set_ms": conv_ms,
        "share_of_step": share, "section_ms": {"conv1": sec_ms[0], "tensor_core_convs": sec_ms[1], "tail": sec_ms[2]},
        "per_launch_ms_event_bracketed": [round(x, 5) for x in per_launch_ms],
        "in_production": {"achieved": overlapped, "frac": overlapped / peak,
                          "frac_of_sustained_peak": (overlapped / peaks["tflops_sustained"]) if peaks.get("tflops_sustained") else None,
                          "how": f"same FLOPs / measured ms_per_step ({args.lanes} forwards in flight; the whole step is charged to the convs)"},
        "peak_source": peaks["source"] + " burst",
    }
    cpu_baseline = None
    if world == 1 and not args.no_cpu_baseline:
        sd = {k: v.detach().cpu() for k, v in model.state_dict().items()}
        threads = pick_cpu_threads(sd, T)
        v, n_it, el = cpu_forward_timer(sd, B, T, budget_s=12.0, threads=threads)
        cpu_baseline = {"value": v, "unit": "emb/s", "cores": threads, "host_cpus": os.cpu_count(),
                        "kind": "port",
                        "sample": f"{n_it} forwards of the same batch-{B} workload in {el:.1f} s (oracle port of "
                                  f"model.py:185-218, torch CPU fp32)"}
    cfg = workload_config(args, world)
    line = {
        "metric": METRIC, "value": value, "unit": "emb/s", "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": args.dtype, "data": "synthetic", "config": cfg,
        "engine": {"forwards_in_flight": args.lanes,
                   "operands": f"{args.dtype} tensor-core operands (BASELINE names bf16: same width and tensor-pipe rate; bf16 "
                               f"misses the 1e-3 parity bar, --dtype bf16 runs it), fp32 accumulate/BN/fc/norm"},
        "timing": "one window of exactly `steps` steps after `warmup` untimed steps, bracketed by barrier + synchronize, "
                  "CUDA events, max over ranks; the launching stream is held ~10 ms before the first event so that the "
                  "first steps are queued when the window opens",
        "clocks": clocks,
        "host_enqueue_ms_per_step": host_ms_value,
        "e2e": {"value": e2e_value, "unit": "emb/s", "h2d_bytes_per_step": in_bytes, "d2h_bytes_per_step": B * 512 * 4,
                "ms_per_step": ms_e2e / K, "host_enqueue_ms_per_step": host_ms_e2e, "api": "EmbeddingPipeline.embed(pinned host batch) -> pinned host embeddings (native dsk_pipeline_submit): H2D, "
                                                  f"the engine forward ({args.lanes} lanes, one CUDA graph per forward) and D2H on their own streams"},
        "gpu_launches": 15 * K,
        "roofline": roofline,
        "tflops_whole_step": B * FLOP_PER_EMB / (ms / K * 1e-3) / 1e12,
    }
    if cpu_baseline:
        line["cpu_baseline"] = cpu_baseline
    return line


def bench_other_dtype(args, D, outputs):
    """The same headline workload with the OTHER 16-bit operand format (bf16 when the line is fp16): BASELINE names bf16,
    the engine defaults to fp16 because bf16 misses the 1e-3 parity bar (DESIGN.md §2); both run at the same tensor-pipe
    rate, and this record keeps the bf16 number beside the headline.  value only (inputs resident), same timing."""
    import torch

    from deepspeaker_pytorch_b200 import EmbeddingPipeline

    other = "bf16" if args.dtype == "fp16" else "fp16"
    dev, B, T, K = D.dev, args.batch, args.frames, args.steps
    model = make_model(other, dev)
    nbuf = L2_BYTES // (B * T * 64 * 4) + 8
    g = torch.Generator(device=dev).manual_seed(7 + D.rank)
    xs = [torch.randn(B, 1, T, 64, device=dev, generator=g) for _ in range(nbuf)]
    pipe = EmbeddingPipeline(model, lanes=args.lanes)
    cur = torch.cuda.current_stream(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    cnt = [0]
    last = [None]
    with torch.no_grad():
        for i in range(2 * args.lanes + args.warmup):
            pipe.embed_device(xs[i % nbuf])
        pipe.synchronize()

        def window():
            D.barrier()
            hold(cur)
            e0.record(cur)
            for _ in range(K):
                last[0] = pipe.embed_device(xs[cnt[0] % nbuf])
                cnt[0] += 1
            for st in pipe.lanes:
                cur.wait_stream(st)
            e1.record(cur)
            D.barrier()
            return e0.elapsed_time(e1)

        ms = timed_window(D, window)
    outputs["other_dtype_embeddings"] = last[0].cpu().numpy()
    return {"dtype": other, "value": D.world * B * K / (ms * 1e-3), "unit": "emb/s", "ms_per_step": ms / K, "steps": K,
            "parity": "eval embeddings ~3e-3 vs the fp32 reference (bar 1e-3)" if other == "bf16" else "eval embeddings 4e-4 - 7e-4 (bar 1e-3)"}


def bench_allpairs(args, D, outputs):
    """BASELINE configs[3]: 1024-utterance all-pairs distance matrix + top-8 hard-negative select (single GPU,
    launch-latency bound: reported in microseconds).  No reference implementation exists (SURVEY §0 fact 3); the
    CPU figure beside it is the oracle's C restatement (oracle/dsk_oracle.c) on one core."""
    import torch

    from deepspeaker_pytorch_b200 import allpairs_topk

    dev = D.dev
    N, Dm, k = 1024, 512, 8
    g = torch.Generator(device=dev).manual_seed(3)
    sets = []
    for _ in range(8):
        E = torch.randn(N, Dm, device=dev, generator=g)
        sets.append(10.0 * E / E.norm(dim=1, keepdim=True))
    labels = (torch.arange(N, device=dev) // 16).long()
    K, W = args.steps, args.warmup
    for i in range(W):
        allpairs_topk(sets[i % 8], labels, k)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    last = [None]

    def window():
        torch.cuda.synchronize()
        hold(torch.cuda.current_stream())
        e0.record()
        for i in range(K):
            last[0] = allpairs_topk(sets[i % 8], labels, k)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1)

    us = window() / K * 1e3
    outputs["allpairs_idx"], outputs["allpairs_val"] = (t.cpu().numpy() for t in last[0])
    # algorithmic bytes: read E (N x D fp32) + labels, write idx (int64) + val (fp32); flops: N*N*D MACs of the Gram
    alg_bytes = N * Dm * 4 + N * 8 + N * k * 12
    peaks = load_peaks()
    rec = {"metric": "microseconds per 1024-utterance all-pairs distance + top-8 select", "value": us, "unit": "us",
           "steps": K, "warmup": W, "higher_is_better": False, "dtype": "f32 (fp16 tensor-core Gram + exact fp32 refinement)",
           "config": {"workload": "1024 x 512 embeddings (norm 10), 64 speakers x 16, k=8, different-speaker candidates "
                                  "(BASELINE configs[3])", "result": "bit-identical indices and distances to the all-fp32 path and the C oracle"},
           "gflops": 2.0 * N * N * Dm / (us * 1e-6) / 1e9,
           "roofline": {"bound": "launch latency (1 GFLOP, 2 MB: neither HBM nor the tensor pipe can be approached)",
                        "achieved": alg_bytes / (us * 1e-6) / 1e9, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                        "frac": alg_bytes / (us * 1e-6) / 1e9 / peaks["hbm_gbs"], "traffic": None},
           "gpu_launches": None}
    if not args.no_cpu_baseline:
        try:
            from oracle import c_oracle

            E0 = sets[0].cpu().numpy()
            lab = labels.cpu().numpy()
            c_oracle.allpairs_topk(E0, lab, k)
            t0 = time.perf_counter()
            n = 0
            while time.perf_counter() - t0 < 3.0:
                c_oracle.allpairs_topk(E0, lab, k)
                n += 1
            cpu_us = (time.perf_counter() - t0) / n * 1e6
            rec["cpu_baseline"] = {"value": cpu_us, "unit": "us", "cores": 1, "kind": "port",
                                   "sample": f"{n} runs of the same 1024 x 512 problem through oracle/dsk_oracle.c (scalar C, one core)"}
        except Exception as e:  # the oracle is test infrastructure: its absence must not break the bench line
            rec["cpu_baseline"] = {"unavailable": str(e)[:200]}
    return rec


TRAIN_FLOP_PER_UTT = 6911819776     # BASELINE.md §2 (forward + backward)


def bench_train(args, D, outputs):
    """BASELINE configs[2] (N=1) / configs[4] (N=8): triplet training step restating train_triplet.py:215-224 with the
    drop-in classes — three train-mode forwards of 128 utterances (issued together through forward_triplet: identical
    results, the three calls and their backwards overlap on three streams), TripletMarginLoss, backward, ONE gradient
    allreduce over the flat bucket (N > 1, NCCL over NVLink), fused Adagrad step (train_triplet.py:369-383)."""
    import torch

    from deepspeaker_pytorch_b200 import FusedAdagrad, TripletMarginLoss
    from deepspeaker_pytorch_b200.parallel import broadcast_parameters, path_parameters

    dev, world, rank = D.dev, D.world, D.rank
    B, T = 128, args.frames
    K, W = args.steps, args.warmup
    model = make_model(args.dtype, dev).train()
    broadcast_parameters(model)
    opt = FusedAdagrad(path_parameters(model), lr=0.1, lr_decay=1e-4, weight_decay=0.0)   # train_triplet.py:70-77,378-382
    crit = TripletMarginLoss(0.1)
    g = torch.Generator(device=dev).manual_seed(100 + rank)
    nset = 48   # 755 MB of distinct triplet batches: with a handful the lr-0.1 steps memorise them and the hinge goes to exactly 0
    xs = [tuple(torch.randn(B, 1, T, 64, device=dev, generator=g) for _ in range(3)) for _ in range(nset)]

    def step(xa, xp, xn):
        out_a, out_p, out_n = model.forward_triplet(xa, xp, xn)     # :215, the three calls in flight together
        loss = crit.forward(out_a, out_p, out_n)                    # :219
        opt.zero_grad()                                             # :222
        loss.backward()                                             # :223
        opt.allreduce()                                             # the one collective of the step
        opt.step()                                                  # :224
        return loss, (out_a, out_p, out_n)

    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for i in range(W):
        step(*xs[i % nset])
    cnt = [0]

    def window():
        D.barrier()
        hold(torch.cuda.current_stream(dev))
        e0.record()
        for _ in range(K):
            last[0] = step(*xs[cnt[0] % nset])
            cnt[0] += 1
        e1.record()
        D.barrier()
        return e0.elapsed_time(e1)

    last = [None]
    ms = timed_window(D, window) / K
    loss, outs = last[0]
    loss_value = float(loss.item())    # loss of the last timed step (48 distinct batches: no memorisation)
    # what the step hands back (loss, the three embedding batches) and what it changed: the updated parameters, as a fixed
    # sample of the flat trained parameters
    flat = torch.cat([p.detach().reshape(-1) for p in path_parameters(model)])
    pick = torch.randint(flat.numel(), (1 << 16,), generator=torch.Generator().manual_seed(0)).to(dev)
    outputs["train_loss"] = loss.detach().reshape(1).cpu().numpy()
    outputs["train_embeddings"] = torch.stack([o.detach() for o in outs]).cpu().numpy()
    outputs["train_params_sample"] = flat[pick].cpu().numpy()
    # e2e: pinned host inputs copied in (on a copy stream, one batch ahead of the step that consumes it - the prefetch any
    # input pipeline does; every step's 15.7 MB still crosses PCIe inside the timed region), loss read back, every step
    nh = 4
    xh = [tuple(torch.randn(B, 1, T, 64).pin_memory() for _ in range(3)) for _ in range(nh)]
    xd = [tuple(torch.empty(B, 1, T, 64, device=dev) for _ in range(3)) for _ in range(2)]
    lh = torch.empty(1).pin_memory()
    copy_stream = torch.cuda.Stream(dev)
    ready = [torch.cuda.Event() for _ in range(2)]
    freed = [torch.cuda.Event() for _ in range(2)]
    cur = torch.cuda.current_stream(dev)

    def stage(slot, k):
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(freed[slot])          # the step that last read this device slot has finished
            for d, h_ in zip(xd[slot], xh[k % nh]):
                d.copy_(h_, non_blocking=True)
            ready[slot].record(copy_stream)

    def window_e2e():
        D.barrier()
        hold(cur)
        for ev in freed:
            ev.record(cur)
        e0.record()
        stage(0, cnt[0])
        for j in range(K):
            slot = j % 2
            if j + 1 < K:
                stage((j + 1) % 2, cnt[0] + 1)
            cur.wait_event(ready[slot])
            loss, _ = step(*xd[slot])
            freed[slot].record(cur)
            lh.copy_(loss.detach().reshape(1), non_blocking=True)
            cnt[0] += 1
        e1.record()
        D.barrier()
        return e0.elapsed_time(e1)

    ms2 = timed_window(D, window_e2e) / K
    if rank != 0:
        return None
    peaks = load_peaks()
    utt_per_step = 3 * B * world
    achieved = 3 * B * TRAIN_FLOP_PER_UTT / (ms * 1e-3) / 1e12     # per GPU
    rec = {"metric": "utterances/sec through the triplet training step (3 forwards + loss + backward + allreduce + Adagrad)",
           "value": utt_per_step / (ms * 1e-3), "unit": "utt/s", "n_gpus": world, "steps": K, "warmup": W,
           "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "dtype": args.dtype,
           "config": {"workload": f"triplet training step, batch {B} triplets per GPU (anchor/pos/neg), synthetic 64x{T} fbank, "
                                  f"branch A (train_triplet.py:215-224), Adagrad lr 0.1 (BASELINE configs[{2 if world == 1 else 4}])",
                      "global_batch_triplets": B * world,
                      "parallelism": f"dp{world}: one NCCL allreduce of 46.5 MB per step" if world > 1 else "single GPU",
                      "l2": "three fresh 5 MB input batches per step (48 distinct triplet batches); ~2 GB of saved activations per step exceed L2"},
           "e2e": {"value": utt_per_step / (ms2 * 1e-3), "unit": "utt/s", "h2d_bytes_per_step": 3 * B * T * 64 * 4,
                   "d2h_bytes_per_step": 4, "ms_per_step": ms2},
           "roofline": {"bound": "tensor", "achieved": achieved, "peak": peaks["tflops_burst"], "unit": "TFLOP/s",
                        "frac": achieved / peaks["tflops_burst"], "traffic": None,
                        "kernel": "whole training step per GPU (forward + dgrad + wgrad convs dominate): 384 utterances x 6 911 819 776 FLOP",
                        "peak_source": peaks["source"] + " burst"},
           "last_loss": loss_value}
    if world == 1 and not args.no_cpu_baseline:
        rec["cpu_baseline"] = cpu_train_baseline(model, T)
    return rec


def cpu_train_baseline(model, T, budget_s=12.0, Bc=8):
    """The reference's training step on host cores (oracle port of train_triplet.py:215-224 + torch.optim.Adagrad),
    on a bounded sample: Bc triplets per step instead of 128 (BASELINE.md §3)."""
    import torch

    from oracle import rescnn_oracle as O

    sd = {k: v.detach().cpu().clone() for k, v in model.state_dict().items() if "classifier" not in k}
    threads = min(os.cpu_count() or 1, 32)
    torch.set_num_threads(threads)
    xs = [O.make_input(Bc, T, seed=s) for s in (0, 1, 2)]
    params = [v for k, v in sd.items() if v.dtype.is_floating_point and "running" not in k]
    n, t0 = 0, None
    while True:
        loss, grads, *_ = O.triplet_step_branch_a(sd, *xs, 0.1)
        with torch.no_grad():   # Adagrad arithmetic on the host (cost is negligible next to the convs)
            for k, g_ in grads.items():
                if g_ is not None:
                    sd[k] = sd[k] - 0.1 * g_ / (g_.abs() + 1e-10)
        if t0 is None:
            t0 = time.perf_counter()   # first step = warm-up
            continue
        n += 1
        el = time.perf_counter() - t0
        if el > budget_s or n >= 20:
            break
    return {"value": 3 * Bc * n / el, "unit": "utt/s", "cores": threads, "host_cpus": os.cpu_count(), "kind": "port",
            "sample": f"{n} steps of {Bc} triplets (3 x {Bc} utterances, forward + backward + update) in {el:.1f} s: oracle port of "
                      f"train_triplet.py:215-224 on torch CPU fp32"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--dtype", default="fp16", choices=["fp16", "bf16"])
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--frames", type=int, default=160)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--lanes", type=int, default=3, help="forwards in flight (compute streams) in the inference pipeline")
    ap.add_argument("--workload", default="all", choices=["all", "infer", "train", "allpairs"],
                    help="all (default): the headline line (batch-64 embedding inference, BASELINE configs[1]) carrying "
                         "`train` (configs[2]/[4]) and `allpairs` (configs[3]) sub-records; infer/train/allpairs: that workload alone")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what each workload's last timed step computed (rank 0) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs saves the outputs of our arm; --impl reference times a shrinking sample of the batch")
    args.warmup = max(args.warmup, 3)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    # stdout carries exactly ONE JSON line: libraries that write to fd 1 (NCCL prints its version banner there)
    # are routed to stderr until the result is printed
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    # the data-parallel allreduce rides NVLink only (north star): no InfiniBand / socket transport on the one box
    # (NCCL_P2P_LEVEL is left to NCCL: forcing "NVL" made it drop to shared-memory transport on a 2-GPU lease whose
    #  topology it does not report as NVLink - 9.25 ms instead of 7.4 ms per training step)
    os.environ.setdefault("NCCL_IB_DISABLE", "1")
    import torch
    import torch.distributed as dist

    assert torch.cuda.is_available(), "bench.py (our arm) needs a GPU; there is no CPU fallback"
    torch.cuda.set_device(local_rank)
    D = Dist(rank, world, local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=D.dev)

    line = None
    outputs = {}
    if args.workload in ("all", "infer"):
        line = bench_infer(args, D, outputs)
    if args.workload in ("all", "train"):
        rec = bench_train(args, D, outputs)
        if rank == 0:
            if line is None:
                line = dict(rec, vs_baseline=None, data="synthetic")
            else:
                line["train"] = rec
    if args.workload == "all" and world == 1:
        line["other_operand_dtype"] = bench_other_dtype(args, D, outputs)
    if args.workload in ("all", "allpairs") and rank == 0:
        rec = bench_allpairs(args, D, outputs)
        if line is None:
            line = dict(rec, n_gpus=1, ms_per_step=rec["value"] / 1e3, scaling="weak", vs_baseline=None, data="synthetic",
                        e2e={"value": rec["value"], "unit": "us", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0})
        else:
            line["allpairs"] = rec
    if rank == 0 and args.dump_outputs:
        write_outputs(args.dump_outputs, outputs)
    if rank == 0:
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
