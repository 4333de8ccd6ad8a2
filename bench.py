#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200-native Silero-VAD engine.

Metric (BASELINE.json): chunks/sec, one chunk = 512 samples @ 16 kHz (256 @ 8 kHz with --sr 8000).
Workload at N=1 (BASELINE.json configs[2]): batch=4096 independent 16 kHz streams, T chunks each (default 64:
537 MB of fp32 audio per step, larger than the 126 MB L2, so nothing is served from cache between steps).
A "step" is one pass of the fused kernel over that batch.  N>1: every rank owns its own 4096 streams
(weak scaling, streams are independent units) and the per-chunk probabilities are all-gathered over NCCL.

  python bench.py --gpus 1 --steps 20 --warmup 3            own arm  (GPU, device-resident inputs + e2e)
  python bench.py ... --dump-outputs DIR                    also write the last timed step's probabilities to DIR/probs.npy
                                                            (seeded inputs: the same arguments give the same inputs on every run)
  python bench.py --impl reference ...                      reference arm: the UNMODIFIED reference (baseline/_ref, TorchScript
                                                            model, audio_forward) on the host cores

Prints ONE JSON line (rank 0).  Keys: see the task contract.  `roofline` is the HBM roofline of the fused kernel
(algorithmic bytes 2052 B/chunk = 2048 B audio + 4 B probability) against MEASURED_PEAKS.json; the path is compute-bound by
~30x (DESIGN.md), so the binding roofline -- the tensor pipe -- is reported beside it as `roofline.tensor`.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

REPO = Path(__file__).resolve().parent
sys.path.insert(0, str(REPO))

ALGO_BYTES = {16000: 2052, 8000: 1028}          # SURVEY.md 8(d): audio fp32 in + prob fp32 out, per chunk
ALGO_FLOP = {16000: 0.730e6, 8000: 0.553e6}     # algorithmic minimum FLOP per chunk (rFFT, dead taps skipped)
HBM_FALLBACK_GBS = 6650.0                       # B200_PROFILING.md fallback when MEASURED_PEAKS.json is absent
BF16_FALLBACK_TFLOPS = 2250.0                   # nominal dense bf16 peak when MEASURED_PEAKS.json is absent
# MACs per chunk that run on tcgen05.  tc kernel: the four convolutions + LSTM (the Nyquist bin and the head stay on CUDA cores);
# h16 kernel: the same plus the STFT as a dense windowed-DFT basis product (N x N per frame, 4 frames).
TENSOR_MAC = {"tc": {16000: 352256, 8000: 270336},
              "h16": {16000: 352256 + 4 * 256 * 256, 8000: 270336 + 4 * 128 * 128}}
KERNEL_INFO = {
    "h16": ("svad_fused_h16 (tcgen05 kind::f16 split precision for STFT + enc0-3 + LSTM, two software-pipelined loops per CTA)", "f16x3",
            "x*w = x_hi*w_hi + x_lo*w_hi + x_hi*w_lo in fp16 (11+11 significand bits per operand) with fp32 accumulate in TMEM; "
            "probabilities within 6e-6 of the fp32 reference on the WAV fixtures"),
    "tc": ("svad_fused_tc (tcgen05 split-TF32 for enc0-3 + LSTM; STFT, gate math and head on the CUDA cores)", "tf32x3",
           "x*w = x_hi*w_hi + x_lo*w_hi + x_hi*w_lo in tf32 with fp32 accumulate; probabilities within 7e-6 of the fp32 reference"),
    "fp32": ("svad_fused_fp32 (fp32 FFMA2, CUDA cores only)", "f32", "IEEE fp32"),
}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=4096, help="streams per GPU")
    ap.add_argument("--chunks", type=int, default=64, help="chunks per stream per step")
    ap.add_argument("--sr", type=int, default=16000, choices=[16000, 8000])
    ap.add_argument("--kernel", default="h16", choices=["h16", "tc", "fp32"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the sustained / latency / segment / configs[3] legs")
    ap.add_argument("--dump-outputs", metavar="DIR", type=Path,
                    help="write the probabilities of the last timed step to DIR/probs.npy (float32) for output-by-output comparison of builds")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes what the GPU arm computed (--impl b200)")
    return args


DUMP_LIMIT_BYTES = 63 * 10**6     # --dump-outputs writes at most 64 MB in all, .npy headers included


def dump_outputs(out_dir, probs):
    """probs: float32 numpy [rows, T].  Above DUMP_LIMIT_BYTES a fixed, seeded sample of rows is written, and the row indices beside it
    (probs_rows.npy, float64), so that two runs with the same arguments write the same sample."""
    out_dir.mkdir(parents=True, exist_ok=True)
    probs = np.ascontiguousarray(probs, np.float32)
    max_rows = max(1, DUMP_LIMIT_BYTES // (probs.shape[1] * 4 + 8))
    if probs.shape[0] > max_rows:
        rows = np.sort(np.random.default_rng(0).choice(probs.shape[0], max_rows, replace=False))
        np.save(out_dir / "probs_rows.npy", rows.astype(np.float64))
        probs = probs[rows]
    np.save(out_dir / "probs.npy", probs)


def peaks():
    p = REPO / "MEASURED_PEAKS.json"
    return json.loads(p.read_text()) if p.exists() else {}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 50 ms while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "50"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def __exit__(self, *a):
        if self.proc:
            time.sleep(0.25)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self):
        sm, mx, pw, reasons = [], [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1])); pw.append(float(r[2]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_min_mhz": min(sm), "sm_max_mhz": max(mx), "power_w_max": max(pw), "reasons": sorted(reasons),
                "samples": len(sm)}


# ------------------------------------------------------------------------------------------ host CPU description / binding
def cpu_info():
    model, phys = "?", set()
    try:
        pkg = None
        for line in Path("/proc/cpuinfo").read_text().splitlines():
            if line.startswith("model name"):
                model = line.split(":", 1)[1].strip()
            elif line.startswith("physical id"):
                pkg = line.split(":")[1].strip()
            elif line.startswith("core id"):
                phys.add((pkg, line.split(":")[1].strip()))
    except OSError:
        pass
    aff = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else os.cpu_count()
    return {"model": model, "logical": os.cpu_count(), "physical": len(phys) or None, "affinity": aff}


def bind_to_gpu_node(index):
    """Pin this process to the CPUs of the NUMA node the GPU hangs off (nvmlDeviceGetCpuAffinity), BEFORE any pinned host buffer is
    allocated, so that first-touch places the staging memory next to the GPU's PCIe root.  Returns the CPU count or None."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
        cpus = [64 * w + b for w, word in enumerate(words) for b in range(64) if (int(word) >> b) & 1]
        cpus = [c for c in cpus if c in os.sched_getaffinity(0)]
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        return None
    return None


# ------------------------------------------------------------------------------------------ reference (CPU) legs
def load_reference():
    """The unmodified reference package staged under baseline/_ref (baseline/stage_reference.py); None when absent."""
    ref = REPO / "baseline" / "_ref"
    if not (ref / "silero_vad" / "data" / "silero_vad.jit").exists():
        return None
    if str(ref) not in sys.path:
        sys.path.insert(0, str(ref))
    import silero_vad
    return silero_vad


def median_time(fn, trials=5, warm=1):
    for _ in range(warm):
        fn()
    ts = []
    for _ in range(trials):
        t0 = time.perf_counter(); fn(); ts.append(time.perf_counter() - t0)
    return statistics.median(ts)


def thread_options(info):
    phys = info["physical"] or info["affinity"] or 1
    phys = min(phys, info["affinity"] or phys)
    return sorted({phys, max(1, phys // 2), min(16, phys)})


def reference_jit_throughput(sv, sr, B, T, threads_opts):
    """BASELINE.md B2: reference TorchScript audio_forward (utils_vad.py:94-110) on [B, n*T] R1 noise, all host cores.  The best
    intra-op thread count among `threads_opts` is kept (torch's CPU pool collapses when oversubscribed)."""
    import torch
    n = 512 if sr == 16000 else 256
    rng = np.random.default_rng(17 + sr)
    x = torch.from_numpy((rng.standard_normal((B, n * T)) * 0.03).astype(np.float32))
    model = sv.load_silero_vad()
    best = None
    for th in threads_opts:
        torch.set_num_threads(th)
        dt = median_time(lambda: model.audio_forward(x, sr), trials=3, warm=1)
        if best is None or dt < best[1]:
            best = (th, dt)
    torch.set_num_threads(best[0])
    dt = median_time(lambda: model.audio_forward(x, sr), trials=5, warm=1)
    torch.set_num_threads(1)
    return {"value": B * T / dt, "threads": best[0], "model": model, "x": x,
            "sample": f"{B} streams x {T} chunks (of the step's {B} x 64), N(0,0.03^2) audio; median of 5, best of {threads_opts} threads"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    info = cpu_info()
    sv = load_reference()
    if sv is not None:
        import torch
        Ts = 4
        r = reference_jit_throughput(sv, args.sr, args.batch, Ts, thread_options(info))
        model, x = r["model"], r["x"]
        torch.set_num_threads(r["threads"])
        for _ in range(max(1, min(args.warmup, 3))):
            model.audio_forward(x, args.sr)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            model.audio_forward(x, args.sr)
        dt = time.perf_counter() - t0
        val = args.batch * Ts * args.steps / dt
        kind, cores = "reference", r["threads"]
        impl = "reference TorchScript model (baseline/_ref/silero_vad: load_silero_vad().audio_forward, utils_vad.py:94-110), torch CPU"
        sample = f"{args.batch} streams x {Ts} chunks per step (of {args.batch} x {args.chunks}), N(0,0.03^2) audio"
    else:   # the staged reference did not travel: the C port of the same graph
        o, x, T, Bs, threads = cpu_arm(args, budget_s=4.0)
        for _ in range(max(1, min(args.warmup, 3))):
            o.audio_forward(x, args.sr, nthreads=threads)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            o.audio_forward(x, args.sr, nthreads=threads)
        dt = time.perf_counter() - t0
        val = Bs * T * args.steps / dt
        kind, cores, impl = "port", threads, "C port of the reference graph (oracle/svad_oracle.c), OpenMP over streams"
        sample = f"{Bs} streams x {T} chunks per step (of {args.batch} x {args.chunks}), N(0,0.03^2) audio"
    print(json.dumps({
        "impl": "reference", "metric": "chunks/sec", "value": val, "unit": "chunks/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"batch={args.batch} independent {args.sr} Hz streams x {args.chunks} chunks (bounded CPU sample)",
                   "sr": args.sr, "impl": impl, "cpu": info},
        "cpu_baseline": {"value": val, "unit": "chunks/s", "cores": cores, "kind": kind, "sample": sample, "cpu": info},
        "e2e": {"value": val, "unit": "chunks/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def cpu_arm(args, threads=None, budget_s=6.0):
    """The reference's algorithm as the C oracle port (oracle/svad_oracle.c, OpenMP over streams): a secondary CPU figure."""
    from oracle.oracle import Oracle
    o = Oracle()
    threads = threads or o.best_threads(args.sr)
    n = 512 if args.sr == 16000 else 256
    rng = np.random.default_rng(17 + args.sr)
    Bs = min(args.batch, 32 * threads)
    x = (rng.standard_normal((Bs, n * 4)) * 0.03).astype(np.float32)
    o.audio_forward(x, args.sr, nthreads=threads)
    t0 = time.perf_counter(); o.audio_forward(x, args.sr, nthreads=threads); dt = time.perf_counter() - t0
    rate = Bs * 4 / max(dt, 1e-6)
    T = int(max(4, min(args.chunks, budget_s * rate / Bs)))
    x = (rng.standard_normal((Bs, n * T)) * 0.03).astype(np.float32)
    return o, x, T, Bs, threads


def cpu_baseline_block(args, dev):
    """`cpu_baseline` of the GPU arm: the reference itself on this box (B2 at the bench batch, all cores; B1 at batch 1, one thread;
    B4 = the reference module moved to the B200, its only GPU path: tuning/tune.py:38), plus the C port as a secondary figure."""
    import torch
    info = cpu_info()
    sr = args.sr
    n = 512 if sr == 16000 else 256
    out = {"unit": "chunks/s", "cpu": info}
    sv = load_reference()
    if sv is not None:
        r = reference_jit_throughput(sv, sr, args.batch, 4, thread_options(info))
        out.update({"value": r["value"], "cores": r["threads"], "kind": "reference", "sample": r["sample"],
                    "what": "reference TorchScript audio_forward (utils_vad.py:94-110), batch = the bench batch, torch CPU"})
        model = r["model"]
        torch.set_num_threads(1)
        T1 = 300
        x1 = torch.from_numpy((np.random.default_rng(5).standard_normal(n * T1) * 0.03).astype(np.float32))

        def b1():
            model.reset_states()
            with torch.no_grad():
                for t in range(T1):
                    model(x1[t * n:(t + 1) * n], sr).item()
        dt = median_time(b1, trials=5, warm=1)
        out["reference_batch1_1thread"] = {"chunks_per_s": T1 / dt, "us_per_chunk": dt / T1 * 1e6,
                                           "what": "model(chunk, sr).item() per chunk, torch.set_num_threads(1) (model.py:3, utils_vad.py:328)"}
        try:
            gm = sv.load_silero_vad().to(dev)
            xg = x1.to(dev)

            def g1():
                gm.reset_states()
                with torch.no_grad():
                    for t in range(T1):
                        gm(xg[t * n:(t + 1) * n], sr).item()
            dt = median_time(g1, trials=3, warm=1)
            Bg, Tg = args.batch, 16
            xb = torch.randn(Bg, n * Tg, device=dev) * 0.03

            def g2():
                gm.reset_states()
                with torch.no_grad():
                    for t in range(Tg):
                        gm(xb[:, t * n:(t + 1) * n], sr)
                torch.cuda.synchronize()
            dtb = median_time(g2, trials=5, warm=2)
            out["reference_on_b200"] = {"batch1_us_per_chunk": dt / T1 * 1e6, "batch_chunks_per_s": Bg * Tg / dtb, "batch": Bg,
                                        "what": "the reference TorchScript module moved to the B200 (tuning/tune.py:38), per-chunk calls, device-resident audio"}
        except Exception as e:   # noqa: BLE001
            out["reference_on_b200"] = {"unavailable": str(e)[:200]}
    o, xs, Ts, Bs, threads = cpu_arm(args)
    t0 = time.perf_counter(); o.audio_forward(xs, sr, nthreads=threads); dt = time.perf_counter() - t0
    port = {"value": Bs * Ts / dt, "unit": "chunks/s", "cores": threads, "kind": "port",
            "sample": f"{Bs} streams x {Ts} chunks, same recipe; C port of the reference graph (oracle/svad_oracle.c)"}
    if sv is None:
        out.update(port)
    else:
        out["port"] = port
    return out


# ------------------------------------------------------------------------------------------ GPU arm
def run_b200(args):
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    numa_cpus = bind_to_gpu_node(local) if world > 1 else None   # before torch allocates pinned memory
    import torch
    import torch.distributed as dist
    from silero_vad_b200 import load_silero_vad

    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl b200 needs a GPU (no CPU fallback)")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    model = load_silero_vad(device=local)
    eng = model.engine
    eng.set_kernel(args.kernel)
    sr, B, T = args.sr, args.batch, args.chunks
    n = 512 if sr == 16000 else 256
    L = n * T
    g = torch.Generator(device=dev); g.manual_seed(17 + sr + rank)
    x = torch.randn(B, L, device=dev, generator=g) * 0.03          # recipe R1 (examples/onnx_sequence/run.py:159-162)
    probs = [torch.empty(B, T, device=dev) for _ in range(2)]       # double-buffered: the gather of step i overlaps the kernel of step i+1
    gathered = [torch.empty(world * B, T, device=dev) for _ in range(2)] if world > 1 else None
    stream = torch.cuda.current_stream().cuda_stream

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def run_steps(k, events=None):
        """k launches; with N > 1 the all-gather of step i is asynchronous (NCCL's own stream) and waited for two steps later, when
        its buffers are reused -- the collective never sits between two kernels."""
        works = [None, None]
        for i in range(k):
            b = i & 1
            if works[b] is not None:
                works[b].wait()
            if events:
                events[i][0].record()
            eng.forward_device(sr, B, L, L, x.data_ptr(), 0, 0, 0, 0, probs[b].data_ptr(), T, stream)
            if events:
                events[i][1].record()
            if world > 1:
                works[b] = dist.all_gather_into_tensor(gathered[b], probs[b], async_op=True)
        for w in works:
            if w is not None:
                w.wait()

    run_steps(max(args.warmup, 3))
    barrier()
    launches0 = eng.launch_count
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    with ClockSampler(local) as clk:
        barrier()
        ev0.record()
        run_steps(args.steps, kev)
        ev1.record()
        barrier()
    ms_total = ev0.elapsed_time(ev1)
    kernel_ms = float(np.mean([a.elapsed_time(b) for a, b in kev]))
    launches = eng.launch_count - launches0
    if world > 1:
        t = torch.tensor([ms_total], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total = float(t.item())
        # what the timed region gathered is what the kernels produced: every rank's block of the last step, checked on every rank
        last = (args.steps - 1) & 1
        assert torch.equal(gathered[last][rank * B:(rank + 1) * B], probs[last]), "all-gather returned something else than this rank's probabilities"
        chk = torch.stack([gathered[last][r * B:(r + 1) * B].sum(dtype=torch.float64) for r in range(world)])
        ref = torch.zeros(world, device=dev, dtype=torch.float64); ref[rank] = probs[last].sum(dtype=torch.float64)
        dist.all_reduce(ref)
        assert torch.equal(chk, ref), "gathered blocks differ from the owners' results"
    if args.dump_outputs and rank == 0:
        last = (args.steps - 1) & 1
        dump_outputs(args.dump_outputs, (gathered if world > 1 else probs)[last].cpu().numpy())
    chunks_per_step = B * T * world
    value = chunks_per_step * args.steps / (ms_total * 1e-3)

    # ---- e2e: host buffers (pinned), H2D + kernel + D2H every step, through the C ABI host entry point
    e2e = None
    if not args.no_e2e:
        xh = x.cpu().pin_memory()
        ph = torch.empty(B, T).pin_memory()
        esteps = args.steps
        for _ in range(2):
            eng.forward_host(sr, B, L, L, xh.data_ptr(), 0, 0, 0, 0, ph.data_ptr(), T)
        barrier()
        t0 = time.perf_counter()
        for _ in range(esteps):
            eng.forward_host(sr, B, L, L, xh.data_ptr(), 0, 0, 0, 0, ph.data_ptr(), T)
        barrier()
        dt = time.perf_counter() - t0
        if world > 1:
            t = torch.tensor([dt], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt = float(t.item())
        assert torch.equal(ph, probs[(args.steps - 1) & 1].cpu()), "host entry point disagrees with device entry point"
        e2e = {"value": chunks_per_step * esteps / dt, "unit": "chunks/s", "h2d_bytes_per_step": B * L * 4, "d2h_bytes_per_step": B * T * 4,
               "ms_per_step": dt / esteps * 1e3, "numa_bound_cpus": numa_cpus,
               "api": "svad_forward_host (C ABI): fp32 host audio in pinned memory, time-sliced H2D overlapped with the kernel, D2H of probabilities"}
        # same call with int16 PCM host audio (what WAV files hold): half the PCIe bytes, bit-identical probabilities
        xi = (xh * 32768.0).round().clamp(-32768, 32767).to(torch.int16).pin_memory()
        pi = torch.empty(B, T).pin_memory()
        for _ in range(2):
            eng.forward_host_pcm16(sr, B, L, L, xi.data_ptr(), 0, 0, 0, 0, pi.data_ptr(), T)
        barrier()
        t0 = time.perf_counter()
        for _ in range(esteps):
            eng.forward_host_pcm16(sr, B, L, L, xi.data_ptr(), 0, 0, 0, 0, pi.data_ptr(), T)
        barrier()
        dti = time.perf_counter() - t0
        if world > 1:
            t = torch.tensor([dti], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dti = float(t.item())
        e2e["pcm16"] = {"value": B * T * world * esteps / dti, "unit": "chunks/s", "h2d_bytes_per_step": B * L * 2, "ms_per_step": dti / esteps * 1e3}

    extra = {}
    if not args.no_extra:
        # ---- sustained leg: >= 2 s of back-to-back launches (the 20-step timed region above is a ~40 ms burst)
        with ClockSampler(local) as sclk:
            barrier()
            s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            nsus = max(args.steps, int(2.2e3 / max(ms_total / args.steps, 1e-3)))
            s0.record()
            run_steps(nsus)
            s1.record()
            barrier()
        sus_ms = s0.elapsed_time(s1)
        if world > 1:
            t = torch.tensor([sus_ms], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            sus_ms = float(t.item())
        extra["sustained"] = {"value": chunks_per_step * nsus / (sus_ms * 1e-3), "unit": "chunks/s", "steps": nsus, "seconds": sus_ms * 1e-3,
                              "clocks": sclk.summary()}
        if world > 1:
            # ---- BASELINE configs[3] as written: 8192 streams per GPU (65 536 at N = 8), and a strong-scaling leg (65 536 streams in total)
            for name, Bx in (("configs3_8192_per_gpu", 8192), ("strong_65536_total", 65536 // world)):
                xx = torch.randn(Bx, L, device=dev, generator=g) * 0.03
                pp = torch.empty(Bx, T, device=dev)
                gg = torch.empty(world * Bx, T, device=dev)
                for _ in range(3):
                    eng.forward_device(sr, Bx, L, L, xx.data_ptr(), 0, 0, 0, 0, pp.data_ptr(), T, stream)
                barrier()
                a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a0.record()
                w = None
                for _ in range(10):
                    if w is not None:
                        w.wait()
                    eng.forward_device(sr, Bx, L, L, xx.data_ptr(), 0, 0, 0, 0, pp.data_ptr(), T, stream)
                    w = dist.all_gather_into_tensor(gg, pp, async_op=True)
                w.wait()
                a1.record()
                barrier()
                t = torch.tensor([a0.elapsed_time(a1)], device=dev, dtype=torch.float64)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                extra[name] = {"value": Bx * T * world * 10 / (float(t.item()) * 1e-3), "unit": "chunks/s", "streams_per_gpu": Bx,
                               "scaling": "weak" if "configs3" in name else "strong"}
                del xx, pp, gg

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    pk = peaks()
    hbm_peak = float(pk.get("hbm_gbs", HBM_FALLBACK_GBS))
    peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in pk else "fallback (B200_PROFILING.md)"
    clocks = clk.summary()
    achieved_gbs = ALGO_BYTES[sr] * B * T / (kernel_ms * 1e-3) / 1e9
    traffic = None
    tp = REPO / "profiles" / "traffic.json"
    if tp.exists():
        try:
            traffic = json.loads(tp.read_text()).get(f"bytes_per_launch_{sr}_{B}x{T}")
        except Exception:
            traffic = None
    kname, dtype, precision = KERNEL_INFO[args.kernel]
    out = {
        "metric": "chunks/sec", "value": value, "unit": "chunks/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": dtype, "data": "synthetic",
        "config": {"workload": f"batch={B} independent {sr} Hz streams per GPU x {T} chunks per step (BASELINE configs[2])",
                   "sr": sr, "batch_per_gpu": B, "chunks_per_stream": T, "global_streams": B * world,
                   "l2": "inputs (%.0f MB/step/GPU) larger than L2, no flush needed" % (B * L * 4 / 1e6),
                   "parallelism": (f"dp{world}: streams sharded, weights replicated, asynchronous NCCL all-gather of probabilities (double-buffered)"
                                   if world > 1 else "single GPU"),
                   "kernel": kname, "precision": precision},
        "gpu_launches": int(launches),
        "kernel_ms": kernel_ms,
        "clocks": clocks,
        "roofline": {"bound": "hbm", "achieved": achieved_gbs, "peak": hbm_peak, "unit": "GB/s", "frac": achieved_gbs / hbm_peak,
                     "traffic": traffic, "traffic_source": "ncu --set full capture under profiles/ (not this run)", "peak_source": peak_src,
                     "algorithmic_bytes_per_chunk": ALGO_BYTES[sr],
                     "note": "the path is compute-bound (356 FLOP/B against a ridge of ~11): the HBM fraction is a few percent by construction; "
                             "traffic ~= algorithmic bytes is the meaningful HBM statement, roofline.tensor the binding one",
                     "algorithmic_flops_over_cuda_core_peak": ALGO_FLOP[sr] * B * T / (kernel_ms * 1e-3) / (eng.sm_count * 128 * 2 * float(pk.get("sm_max_mhz", 1965.0)) * 1e6)},
    }
    if args.kernel in TENSOR_MAC:
        # what the kernel executes on tcgen05 against the measured dense tensor peak.  Split precision issues 3 products per MAC; tf32
        # runs at half the bf16 / fp16 rate.  MEASURED_PEAKS.json: bf16 burst (kernel timed alone) and sustained (long runs).
        bf16 = float(pk.get("bf16_tflops", BF16_FALLBACK_TFLOPS))
        bf16_sus = float(pk.get("bf16_tflops_sustained", bf16))
        algo_t = 2.0 * TENSOR_MAC[args.kernel][sr] * B * T / (kernel_ms * 1e-3) / 1e12
        rate = 1.0 if args.kernel == "h16" else 0.5
        out["roofline"]["tensor"] = {"bound": "tensor", "achieved": 3.0 * algo_t, "peak": rate * bf16, "unit": "TFLOP/s", "frac": 3.0 * algo_t / (rate * bf16),
                                     "algorithmic_tflops": algo_t,
                                     "peak_source": ("measured (MEASURED_PEAKS.json bf16_tflops, burst" if "bf16_tflops" in pk else "nominal (2.25 PFLOP/s dense bf16")
                                                    + ("; fp16 runs at the bf16 rate)" if args.kernel == "h16" else "; tf32 at half of it)"),
                                     "frac_of_sustained_peak": 3.0 * algo_t / (rate * bf16_sus),
                                     "note": "MACs on tcgen05 x 3 products of the hi/lo split; with 32 streams per CTA (one CTA per SM) an instruction covers 32-128 columns and costs "
                                             "46-64 cycles (tools/umma_f16_unit.cu), i.e. 1/4 - 1/2 of the dense rate: the instruction count, not the FLOP peak, binds"}
    if e2e:
        out["e2e"] = e2e
    out.update(extra)
    if world == 1 and not args.no_extra:
        out["latency_b1"] = latency_b1(eng, sr, dev, stream)
        out["segments"] = segments_leg(sr, probs[0])
    if world == 1 and not args.no_cpu_baseline:
        out["cpu_baseline"] = cpu_baseline_block(args, dev)
    print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


def latency_b1(eng, sr, dev, stream):
    """BASELINE configs[1]: batch = 1 streaming, one 512-sample chunk per call through the stateless C ABI step (host buffers)."""
    import torch
    n1 = 512 if sr == 16000 else 256
    x1 = np.zeros((1, n1 + n1 // 8), np.float32)
    st1 = np.zeros((2, 1, 128), np.float32)
    pr1 = np.zeros(1, np.float32)
    lat = []
    for i in range(400):
        x1[0, n1 // 8:] = np.random.default_rng(i).standard_normal(n1).astype(np.float32) * 0.03
        t0 = time.perf_counter()
        eng.step_host(sr, 1, x1.ctypes.data, st1.ctypes.data, pr1.ctypes.data, st1.ctypes.data)
        lat.append((time.perf_counter() - t0) * 1e6)
    lat = np.sort(np.asarray(lat[50:]))
    xs = torch.randn(1, n1 * 256, device=dev) * 0.03
    ps = torch.empty(1, 256, device=dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    eng.forward_device(sr, 1, n1 * 256, n1 * 256, xs.data_ptr(), 0, 0, 0, 0, ps.data_ptr(), 256, stream)
    e0.record()
    eng.forward_device(sr, 1, n1 * 256, n1 * 256, xs.data_ptr(), 0, 0, 0, 0, ps.data_ptr(), 256, stream)
    e1.record(); torch.cuda.synchronize()
    out = {"step_host_us_median": float(np.median(lat)), "step_host_us_p99": float(lat[int(0.99 * len(lat))]),
           "kernel_us_per_chunk": e0.elapsed_time(e1) * 1e3 / 256,
           "note": "batch=1 (BASELINE configs[1]): svad_step_host per chunk incl. copies and sync; kernel = 8-CTA cluster kernel, 256 chunks in one launch"}
    if hasattr(eng, "stream_open"):
        out["persistent"] = persistent_latency(eng, sr)
    return out


def persistent_latency(eng, sr):
    """The persistent single-stream kernel fed through mapped host memory (svad_stream_*): per-chunk latency without a launch."""
    n1 = 512 if sr == 16000 else 256
    h = eng.stream_open(sr)
    lat = []
    x = np.zeros(n1, np.float32)
    for i in range(600):
        x[:] = np.random.default_rng(i).standard_normal(n1).astype(np.float32) * 0.03
        t0 = time.perf_counter()
        eng.stream_push(h, x)
        lat.append((time.perf_counter() - t0) * 1e6)
    eng.stream_close(h)
    lat = np.sort(np.asarray(lat[100:]))
    return {"us_median": float(np.median(lat)), "us_p99": float(lat[int(0.99 * len(lat))]),
            "note": "svad_stream_push: chunk written to mapped pinned memory, the persistent cluster kernel polls a mailbox, the probability comes "
                    "back through mapped memory (no launch, no cudaMemcpy, no stream synchronize per chunk)"}


def segments_leg(sr, probs_dev):
    """SURVEY 8(f)-1: the batched timestamp automaton (svad_speech_segments, host threads) on this step's [B, T] probabilities."""
    from silero_vad_b200 import _cabi
    from silero_vad_b200.utils_vad import _segment_params
    p = probs_dev.cpu().numpy()
    B, T = p.shape
    rng = np.random.default_rng(0)
    speechy = np.clip(p + (rng.uniform(size=p.shape) < 0.5) * rng.uniform(0.3, 1.0, size=p.shape), 0, 1).astype(np.float32)   # R1 noise alone never triggers
    n = 512 if sr == 16000 else 256
    lens = np.full(B, T * n, np.int64)
    params = _segment_params(sr, 0.5, None, 250, float("inf"), 100, 30, 98, True)
    segs = _cabi.speech_segments(speechy, lens, params)
    ts = []
    for _ in range(5):
        t0 = time.perf_counter()
        segs = _cabi.speech_segments(speechy, lens, params)
        ts.append(time.perf_counter() - t0)
    dt = statistics.median(ts)
    return {"chunks_per_s": B * T / dt, "ms": dt * 1e3, "segments": int(sum(len(s) for s in segs)),
            "note": "svad_speech_segments (threaded over rows) on the step's probabilities with synthetic speech bursts mixed in, incl. the Python list build"}


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_b200(a)
