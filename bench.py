#!/usr/bin/env python
"""bench.py — headline benchmark of the B200 hot path (contract: see DESIGN.md "Measurement").

One "step" = one pass of the RRC matched-filter FIR sweep (BASELINE.json configs[1]):
real-tap RRC filters of 33, 65, 129 and 257 taps (span 16, sps 2/4/8/16, alpha 0.35) applied as
streaming ComplexFIRFilter.Filter() over 2^28 synthetic complex samples (uniform(-1,1) from the
counter RNG, seed 1), i.e. 4 kernel launches per step.  Inputs (2 GiB) and outputs (2 GiB) are far
larger than the 126 MB L2, so no flush is needed between iterations.

  value   Msamples/s, whole job (all ranks), inputs resident in HBM, CUDA-event timed, max over ranks
  e2e     the same sweep through the host-pointer C ABI call (qpsk_fir_filter) with pinned host
          buffers: H2D + kernel + D2H inside the timed region
  roofline the launch that dominates the step (257 taps: FP32-FMA bound) + one entry per tap count
  cpu_baseline the oracle's C++ restatement of the C# SIMD FIR on the host cores (bounded sample)

`--impl reference` times that CPU restatement alone (the C# reference cannot run here: no .NET).

`--steps` and `--warmup` set the timed and warm-up steps of the FIR sweep, the decimate-by-D leg, the chain and modulator
legs and the host-pointer (e2e) legs.  Fixed in size: the pageable / registered variants (one timed call each), the stream
leg (a fixed 400 blocks through each API) and the CPU baselines (a fixed sample of samples or bursts).

`--dump-outputs DIR` writes, after the timed steps, what each of the four filters returned in the last timed step, so that
two builds run with the same arguments (identical inputs) can be compared output for output: DIR/fir_taps<N>.npy holds
float32 (I, Q) pairs at the output positions listed in DIR/sample_index.npy (float64): the first 4096 outputs (the delay
line carried over from the step before) and a fixed random sample (seed 0) of 2^20 of the others, about 42 MB in all.
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
sys.dont_write_bytecode = True      # the benchmark leaves the source tree as it found it (no __pycache__ of its imports)

TAPS = [(16, 2), (16, 4), (16, 8), (16, 16)]  # (span, sps) -> 33, 65, 129, 257 taps
ALPHA = 0.35
LOG2_SAMPLES = 28
METRIC = "Msamples/s RRC FIR sweep (taps 33-257) on 2^28 cf32 samples"
DUMP_HEAD, DUMP_SAMPLE = 4096, 1 << 20          # outputs per filter kept by --dump-outputs: 4 x ~8 MB of cf32


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f).get("hbm_gbs", 6650.0), "measured"
    return 6650.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "20"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=10)       # reaped here, so no sampler outlives the benchmark
        except subprocess.TimeoutExpired:
            self.proc.kill()
            self.proc.wait()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        # under load = the upper half of the samples (idle samples before/after the region are lower)
        load = sm[len(sm) // 2:] if sm else []
        return {"sm_mhz": (load[len(load) // 2] if load else None), "sm_max_mhz": (max(mx) if mx else None),
                "samples": len(sm), "reasons": sorted(reasons)}


def ncu_traffic():
    """DRAM bytes per launch of the FIR kernel from the committed `ncu --set full` capture (profiles/)."""
    p = os.path.join(ROOT, "profiles", "r02_ncu_traffic.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f)
    return None


def copy_ceiling(torch, hin, hout, n_bytes):
    """Pinned-copy rates of this box (GB/s): H2D alone, D2H alone, both at once.  The host-pointer path moves
    8 B in + 8 B out per complex sample, so `duplex_each / 8 B` is the ceiling of the e2e number."""
    hi = torch.from_numpy(hin.array).view(torch.uint8)[:n_bytes]
    ho = torch.from_numpy(hout.array).view(torch.uint8)[:n_bytes]
    di = torch.empty(n_bytes, dtype=torch.uint8, device="cuda")
    do = torch.empty(n_bytes, dtype=torch.uint8, device="cuda")
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()

    def run(h2d, d2h):
        best = 0.0
        for _ in range(2):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            if h2d:
                with torch.cuda.stream(s1):
                    di.copy_(hi, non_blocking=True)
            if d2h:
                with torch.cuda.stream(s2):
                    ho.copy_(do, non_blocking=True)
            torch.cuda.synchronize()
            best = max(best, n_bytes / (time.perf_counter() - t0) / 1e9)
        return best

    r = {"h2d_gbs": run(True, False), "d2h_gbs": run(False, True), "duplex_each_gbs": run(True, True)}
    del di, do
    return r


def pin_to_gpu_cores(index: int):
    """Bind this rank to the CPU cores NVML reports as local to its GPU (the NUMA node its PCIe root hangs off), so that the
    pinned staging buffers of the host-pointer legs are allocated and copied from local memory.  Best effort."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
        cores = [64 * w + b for w, m in enumerate(words) for b in range(64) if (m >> b) & 1]
        cores = [c for c in cores if c < (os.cpu_count() or 1)]
        if cores:
            os.sched_setaffinity(0, cores)
        return {"cores": len(cores), "first": cores[0] if cores else None, "of": os.cpu_count()}
    except Exception as e:   # noqa: BLE001 - reported in the JSON line
        return {"error": repr(e)[:120]}


def taps_for(orc_or_q, span, sps):
    h = orc_or_q.RRCFilter.generateCoefficents(span, ALPHA, sps * 1000, 1000)
    return orc_or_q.real_taps_to_iq(h)


def cpu_baseline(n_each_log2: int = 20):
    """Oracle port of the C# SIMD FIR (FIRFilter.cs:59-91,144-211) on all host cores: one independent
    stream per core, each 2^n_each_log2 samples per tap count."""
    import numpy as np
    import oracle as O
    O.build()
    cores = os.cpu_count() or 1
    n_each = 1 << n_each_log2
    x = O.fill_uniform(1, 0, 0, 2 * n_each * cores)
    y = np.empty_like(x)
    t_total = 0.0
    per = {}
    for span, sps in TAPS:
        taps = taps_for(O, span, sps)
        t0 = time.perf_counter()
        O.fir_filter_mt(taps, x, y, 2 * n_each, cores)
        dt = time.perf_counter() - t0
        per[taps.size // 2] = n_each * cores / dt / 1e6
        t_total += dt
    # single thread, what the reference library itself uses
    t1 = 0.0
    n1 = 1 << max(n_each_log2 - 1, 10)
    for span, sps in TAPS:
        taps = taps_for(O, span, sps)
        t0 = time.perf_counter()
        O.fir_filter_mt(taps, x, y, 2 * n1, 1)
        t1 += time.perf_counter() - t0
    return {
        "value": len(TAPS) * n_each * cores / t_total / 1e6, "unit": "Msamples/s", "cores": cores, "kind": "port",
        "sample": f"{cores} independent streams x 2^{n_each_log2} samples x taps {{33,65,129,257}}, C++ AVX2 restatement of "
                  f"the C# SIMD FIR (no .NET in this image)",
        "single_thread_value": len(TAPS) * n1 / t1 / 1e6,
        "per_taps": per, "seconds": t_total + t1,
    }


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    t_all, vals = [], []
    for i in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        b = cpu_baseline(22)
        dt = time.perf_counter() - t0
        if i >= args.warmup:
            vals.append(b["value"]); t_all.append(dt)
    v = sum(vals) / len(vals)
    b["value"] = v
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": "Msamples/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * sum(t_all) / len(t_all), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "fir_sweep taps{33,65,129,257} (bounded sample per step: cores x 2^22 samples per tap count)",
                   "same_config": False,
                   "sample_note": "same filters, same input distribution and the same metric as the GPU arm, on a bounded sample: one "
                                  "independent stream of 2^22 samples per host core and tap count instead of one 2^28-sample stream "
                                  "(throughput of this per-sample loop does not depend on the stream length).  All host cores are "
                                  "used; the reference library itself is single-threaded (cpu_baseline.single_thread_value)"},
        "cpu_baseline": b,
        "e2e": {"value": v, "unit": "Msamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--log2-samples", type=int, default=LOG2_SAMPLES)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-chain", action="store_true")
    ap.add_argument("--no-decimate", action="store_true")
    ap.add_argument("--no-scaling-legs", action="store_true", help="skip the 16384-channel strong / saturated chain legs")
    ap.add_argument("--channels-total", type=int, default=16384, help="BASELINE.json configs[3]: size of the fixed channel set")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write a fixed sample of the last timed step's filter outputs to DIR "
                                                            "as .npy (rank 0)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.impl == "reference" and args.dump_outputs:
        ap.error("--dump-outputs writes the GPU filters' outputs; the reference arm has none")
    if args.impl == "reference":
        return run_reference(args)

    import numpy as np
    import torch
    import torch.distributed as dist

    # NCCL_DEBUG / NCCL_DEBUG_FILE are left exactly as the launcher set them (the driver reads the communicator's rank
    # count from that log); the JSON line is printed last, after the process group is gone
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    # N > 1 only: at N = 1 the CPU-baseline legs of the same process use every host core
    affinity = pin_to_gpu_cores(local) if world > 1 else {"cores": os.cpu_count(), "note": "unpinned at N = 1"}
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    from qpsk_modulator_demodulator_b200 import build as qbuild
    if rank == 0:
        qbuild.build()
    if world > 1:
        dist.barrier()
    import qpsk_modulator_demodulator_b200 as Q
    Q.set_device(local)
    build_id = Q._native.build_id()          # lib() already refused a library that is not the build of this tree
    # the library's own NCCL communicator (qpsk_comm_*): what gathers the BER counters; its id travels over torch's store
    comm = None
    if world > 1:
        from qpsk_modulator_demodulator_b200 import shard

        def exchange(ident):
            t = torch.zeros(128, dtype=torch.uint8, device="cuda")
            if ident is not None:
                t.copy_(torch.frombuffer(bytearray(ident), dtype=torch.uint8))
            dist.broadcast(t, 0)
            return bytes(t.cpu().numpy().tobytes())

        comm = shard.CounterComm(world, rank, exchange)

    n = 1 << args.log2_samples
    # an explicit (non-default) stream: a NULL stream handle means "the handle's own stream" in the C ABI,
    # and CUDA events must be recorded on the stream the kernels are launched on
    tstream = torch.cuda.Stream()
    torch.cuda.set_stream(tstream)
    stream = tstream.cuda_stream
    assert stream != 0
    x = torch.empty(2 * n, dtype=torch.float32, device="cuda")
    # one output buffer per filter, so that all four outputs of the last timed step survive it (--dump-outputs)
    ys = [torch.empty(2 * n, dtype=torch.float32, device="cuda") for _ in TAPS]
    y = ys[-1]
    Q.fill_uniform_dev(1, rank, 0, 2 * n, x.data_ptr(), stream)

    def history(nt):
        """The delay line a streaming filter of nt taps carries into its last call over x: the tail of x, or zeros when
        (--warmup 0 --steps 1) that call was its first."""
        tail = x[2 * (n - (nt - 1)):]
        return tail if args.warmup + args.steps > 1 else torch.zeros_like(tail)
    filters = []
    for span, sps in TAPS:
        t = taps_for(Q, span, sps)
        filters.append((t.size // 2, Q.ComplexFIRFilter(t)))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step(ev=None):
        for i, (nt, f) in enumerate(filters):
            if ev is not None:
                ev[i][0].record()
            f.filter_dev(x.data_ptr(), ys[i].data_ptr(), 2 * n, stream=stream)
            if ev is not None:
                ev[i][1].record()

    for _ in range(args.warmup):
        step()
    barrier()
    fma_peak = Q.measure_fma_peak()
    barrier()

    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
        time.sleep(0.3)
    evs = [[(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in filters]
           for _ in range(args.steps)]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    Q.launch_count_reset()
    barrier()
    e0.record()
    for k in range(args.steps):
        step(evs[k])
    e1.record()
    barrier()
    launches = Q.launch_count()
    ms = e0.elapsed_time(e1)
    kernels = {nt: f.last_kernel() for nt, f in filters}     # what the library actually launched for each tap count
    if args.dump_outputs and rank == 0:
        if n <= DUMP_HEAD + DUMP_SAMPLE:
            idx = np.arange(n)
        else:
            rest = np.random.default_rng(0).choice(n - DUMP_HEAD, DUMP_SAMPLE, replace=False) + DUMP_HEAD
            idx = np.concatenate([np.arange(DUMP_HEAD), np.sort(rest)])
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "sample_index.npy"), idx.astype(np.float64))
        idx_dev = torch.from_numpy(idx).cuda()
        for (nt, _), yo in zip(filters, ys):
            np.save(os.path.join(args.dump_outputs, f"fir_taps{nt}.npy"), yo.view(-1, 2).index_select(0, idx_dev).cpu().numpy())
        del idx_dev
    # in-run parity of the timed output: y still holds what the LAST timed launch wrote (the longest filter, delay line carried
    # from the step before = the tail of x).  Two windows — the head of the stream and one across tile seams deep inside — are
    # recomputed by the CPU oracle (checker only) from the same samples; north_star's tolerance 1e-5 * max|y|.
    fir_parity = None
    if rank == 0 and not args.no_cpu:
        import oracle as O
        nt_last, f_last = filters[-1]
        wlen = 4096
        taps_last = taps_for(Q, *TAPS[-1])
        worst, scale = 0.0, 0.0
        for lo in (0, n // 3):
            if lo == 0:
                seg = torch.cat([history(nt_last), x[:2 * wlen]]).cpu().numpy()
            else:
                seg = x[2 * (lo - (nt_last - 1)): 2 * (lo + wlen)].cpu().numpy()
            want = O.ComplexFIRFilter(taps_last).Filter(seg)[2 * (nt_last - 1):]
            got = y[2 * lo: 2 * (lo + wlen)].cpu().numpy()
            worst = max(worst, float(np.abs(got - want).max()))
            scale = max(scale, float(np.abs(want).max()))
        fir_parity = {"launch": f"last timed launch, {nt_last} taps, {kernels[nt_last]}",
                      "windows": f"outputs [0, {wlen}) (delay line carried from the previous step) and [n/3, n/3 + {wlen})",
                      "oracle": "oracle.ComplexFIRFilter.Filter (reference summation order) on the same samples",
                      "max_abs_err_over_max_abs": worst / max(scale, 1e-30), "tolerance": 1e-5,
                      "ok": bool(worst <= 1e-5 * scale)}
    clk = clocks.stop() if rank == 0 else None
    t_ms = torch.tensor([ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t_ms, op=dist.ReduceOp.MAX)
    ms_max = float(t_ms.item())
    per_ms = [sum(evs[k][i][0].elapsed_time(evs[k][i][1]) for k in range(args.steps)) / args.steps for i in range(len(filters))]

    hbm_peak, peak_src = peaks()
    roofs = []
    for (nt, _), t in zip(filters, per_ms):
        gbs = 16.0 * n / (t * 1e-3) / 1e9
        tf = 4.0 * nt * n / (t * 1e-3) / 1e12
        bound = "hbm" if (16.0 * n / (hbm_peak * 1e9)) >= (4.0 * nt * n / (fma_peak * 1e12)) else "fma"
        roofs.append({"taps": nt, "kernel": kernels[nt], "ms": t, "msamples_s": n / (t * 1e-3) / 1e6, "bound": bound,
                      "hbm_gbs": gbs, "hbm_frac": gbs / hbm_peak, "fma_tflops": tf, "fma_frac": tf / fma_peak,
                      "frac": (gbs / hbm_peak) if bound == "hbm" else (tf / fma_peak)})
        if "split2" in kernels[nt]:
            # fir_split2_kernel (2-parallel fast-FIR split): (3P+1) half-length sub-filter outputs per 2P = 10 samples, i.e.
            # 16 * G/2 packed FMAs = 3.2*G flop per sample where the direct form (`fma_tflops`, the algorithmic count) needs
            # 4*taps — `frac` above 1 would mean faster than ANY direct-form kernel can run; `executed_frac` is the share of
            # the FP32 peak the launch really kept busy
            g_even = (nt + 1) & ~1
            ex = 3.2 * g_even * n / (t * 1e-3) / 1e12
            roofs[-1].update({"executed_flop_per_sample": 3.2 * g_even, "executed_tflops": ex, "executed_frac": ex / fma_peak})
    tr = ncu_traffic()
    if tr is not None and tr.get("log2_samples") == args.log2_samples:
        for r in roofs:
            t = tr["per_taps"].get(str(r["taps"]))
            if t:
                r["traffic"] = t["traffic"]
                r["algorithmic_bytes"] = 16.0 * n
                # the FMA-pipe activity ncu measured for the same launch: an independent check of `fma_frac`, whose
                # denominator is this run's own FFMA2 micro-benchmark (nominal peak: fma_peak_nominal)
                r["ncu_fma_pipe_active_pct"] = t.get("fma_pipe_active_pct")
                r["fma_frac_of_nominal"] = r["fma_tflops"] / (148 * 128 * 2 * 1.965e9 / 1e12)
    dom = max(roofs, key=lambda r: r["ms"])
    hbm_dom = max((r for r in roofs if r["bound"] == "hbm"), key=lambda r: r["ms"], default=None)
    roofline = {
        "kernel": dom["kernel"], "taps": dom["taps"], "bound": dom["bound"],
        "achieved": dom["hbm_gbs"] if dom["bound"] == "hbm" else dom["fma_tflops"],
        "peak": hbm_peak if dom["bound"] == "hbm" else fma_peak,
        "unit": "GB/s" if dom["bound"] == "hbm" else "TFLOP/s",
        "frac": dom["frac"], "traffic": dom.get("traffic"),
        "traffic_source": (tr["source"] if tr is not None and dom.get("traffic") else None),
        "fma_peak_nominal": 148 * 128 * 2 * 1.965e9 / 1e12,
        "peak_source": (f"HBM {peak_src} (MEASURED_PEAKS.json)" if dom["bound"] == "hbm"
                        else "FP32 FMA peak measured in this run by qpsk_measure_fma_peak (FFMA2 micro-benchmark)"),
        "algorithmic": "16 B and 4*taps flop per complex sample (DESIGN.md)",
    }
    if "executed_frac" in dom:
        roofline.update({"executed_tflops": dom["executed_tflops"], "executed_frac": dom["executed_frac"],
                         "note": "achieved / frac count the direct form's 4*taps flop per sample (the algorithmic work); the "
                                 "fast-FIR split executes 0.8 of them, executed_* is what the FP32 pipe really did"})
    # the same kernel where it is HBM-bound (33 taps), against the driver-measured copy bandwidth
    roofline_hbm = None
    if hbm_dom is not None:
        roofline_hbm = {"kernel": hbm_dom["kernel"], "taps": hbm_dom["taps"], "bound": "hbm", "achieved": hbm_dom["hbm_gbs"],
                        "peak": hbm_peak, "unit": "GB/s", "frac": hbm_dom["hbm_frac"], "traffic": hbm_dom.get("traffic"),
                        "peak_source": f"HBM {peak_src} (MEASURED_PEAKS.json)"}

    # ---- decimate-by-D matched filter (north_star (2); SURVEY §8d): 8 + 8/D B and 4N/D flop per INPUT sample ----------
    decimate = []
    if not args.no_decimate:
        for span, sps, dec in ((16, 2, 2), (16, 4, 2), (16, 8, 2), (16, 4, 4), (16, 8, 8), (16, 16, 16)):
            t = taps_for(Q, span, sps)
            nt = t.size // 2
            f = Q.ComplexFIRFilter(t)
            for _ in range(args.warmup):
                f.decimate_dev(x.data_ptr(), 2 * n, dec, y.data_ptr(), 2 * n, stream=stream)
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            reps = args.steps
            ev0.record()
            for _ in range(reps):
                f.decimate_dev(x.data_ptr(), 2 * n, dec, y.data_ptr(), 2 * n, stream=stream)
            ev1.record()
            torch.cuda.synchronize()
            tms = ev0.elapsed_time(ev1) / reps
            gbs = (8.0 + 8.0 / dec) * n / (tms * 1e-3) / 1e9
            tf = 4.0 * nt / dec * n / (tms * 1e-3) / 1e12
            bound = "hbm" if ((8.0 + 8.0 / dec) / (hbm_peak * 1e9)) >= (4.0 * nt / dec / (fma_peak * 1e12)) else "fma"
            par = None
            if rank == 0 and not args.no_cpu:
                # the timed output against the oracle: first 2048 kept outputs (delay line carried from the previous call = the
                # tail of x; n is a multiple of D, so the kept-output phase is 0) — oracle filter at full rate, every D-th kept
                import oracle as O
                wo = 2048
                seg = torch.cat([history(nt), x[:2 * wo * dec]]).cpu().numpy()
                want = O.decimate(O.ComplexFIRFilter(t).Filter(seg)[2 * (nt - 1):], dec)
                got = y[:2 * wo].cpu().numpy()
                err = float(np.abs(got - want).max() / max(float(np.abs(want).max()), 1e-30))
                par = {"outputs_checked": wo, "max_abs_err_over_max_abs": err, "tolerance": 1e-5, "ok": bool(err <= 1e-5)}
            decimate.append({"taps": nt, "decim": dec, "kernel": f.last_kernel(), "parity": par, "ms": tms, "msamples_s_in": n / (tms * 1e-3) / 1e6,
                             "bound": bound, "hbm_gbs": gbs, "fma_tflops": tf,
                             "frac": gbs / hbm_peak if bound == "hbm" else tf / fma_peak,
                             "algorithmic": "8 + 8/D B and 4*taps/D flop per input sample",
                             "peak_note": "HBM peak = the driver-measured COPY bandwidth (1 B read per B written); these launches "
                                          "read D B per B written, and read-heavy mixes run above the copy figure on this part "
                                          "(a pure fill reaches 7.5 TB/s), so an HBM-bound frac can touch 1.0"})
            del f

    # ---- e2e: host-pointer C ABI with pinned buffers -------------------------------------------
    e2e = None
    if not args.no_e2e:
        hin = Q.PinnedBuffer(2 * n)
        hout = Q.PinnedBuffer(2 * n)
        torch.cuda.synchronize()
        torch.from_numpy(hin.array).copy_(x)  # fill the pinned input from the device copy (untimed)
        torch.cuda.synchronize()
        for _, f in filters:
            f.reset()
        pcie = copy_ceiling(torch, hin, hout, 1 << 30)
        k_e2e = args.steps
        for _, f in filters:                                    # one untimed full step: slot buffers, streams, first DMA
            f.Filter(hin.array, hout.array)
            f.reset()
        barrier()
        step_s = []
        for _ in range(k_e2e):
            t0 = time.perf_counter()
            for _, f in filters:
                f.Filter(hin.array, hout.array)
            torch.cuda.synchronize()
            step_s.append(time.perf_counter() - t0)
        # host<->device copy rates on shared boxes vary from step to step (other tenants on the same PCIe root / host
        # memory): the value is taken on the median step, every step is listed
        t_e = torch.tensor([sorted(step_s)[len(step_s) // 2]], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t_e, op=dist.ReduceOp.MAX)
        dt = float(t_e.item()) * k_e2e
        e2e = {"value": world * k_e2e * len(filters) * n / dt / 1e6, "unit": "Msamples/s",
               "h2d_bytes_per_step": len(filters) * 8 * n, "d2h_bytes_per_step": len(filters) * 8 * n,
               "steps": k_e2e, "api": "qpsk_fir_filter (host pointers, pinned, chunked H2D/kernel/D2H pipeline)",
               "step_ms": [round(1e3 * t, 2) for t in step_s], "timing": "median step (max over ranks)",
               "bound": "pcie", "pinned_copy_gbs": pcie,
               "ceiling": world * pcie["duplex_each_gbs"] * 1e9 / 8.0 / 1e6}
        e2e["frac_of_ceiling"] = e2e["value"] / e2e["ceiling"]
        if world == 1:
            # the same call on memory a C# host really has: a float[] pinned in place (qpsk_host_register on the GCHandle's
            # address) and plain pageable arrays (the driver bounces those through its own staging buffers).  One timed step.
            def one_step(xa, ya):
                for _, f in filters:
                    f.reset()
                filters[0][1].Filter(xa[: 1 << 22], ya[: 1 << 22])      # touch the path once, untimed
                filters[0][1].reset()
                t0 = time.perf_counter()
                for _, f in filters:
                    f.Filter(xa, ya)
                torch.cuda.synchronize()
                return time.perf_counter() - t0
            xa = np.array(hin.array, copy=True)
            ya = np.empty_like(xa)
            ya.fill(0.0)                                                 # every output page resident before the timing (np.zeros maps lazily)
            tp = one_step(xa, ya)
            e2e["pageable"] = {"value": len(filters) * n / tp / 1e6, "unit": "Msamples/s", "steps": 1}
            with Q.RegisteredArray(xa), Q.RegisteredArray(ya):
                tr_ = one_step(xa, ya)
            e2e["registered"] = {"value": len(filters) * n / tr_ / 1e6, "unit": "Msamples/s", "steps": 1,
                                 "api": "qpsk_host_register on the caller's arrays, then qpsk_fir_filter"}
            del xa, ya
        hin.free(); hout.free()

    chain = chain_fll = modulator = stream_leg = None
    if not args.no_chain:
        import bench_chain
        d = dist if world > 1 else None
        torch.cuda.synchronize()
        del y, ys
        torch.cuda.empty_cache()
        cpu_legs = rank == 0 and world == 1 and not args.no_cpu
        # config 3 / config 4's per-GPU share: 2048 channels per GPU (weak: 16384 channels at N = 8).  At N = 1 every
        # channel is replayed through the oracle; at N > 1, 128 channels per rank.
        par = None if world == 1 else 128
        common = dict(steps=args.steps, warmup=args.warmup, hbm_peak=hbm_peak, comm=comm)
        chain = bench_chain.run_chain(Q, torch, d, world, rank, stream, use_fll=False, cpu=cpu_legs, parity_channels=par,
                                      label="weak: 2048 channels per GPU", **common)
        chain_fll = bench_chain.run_chain(Q, torch, d, world, rank, stream, use_fll=True, cpu=cpu_legs, parity_channels=par,
                                          label="weak: 2048 channels per GPU", **common)
        # config 4 proper: the FIXED 16384-channel set sharded over the GPUs (strong scaling: 16384 / N per GPU), and the
        # saturated weak case (16384 channels on every GPU).  At N = 1 the two coincide.
        scaling_legs = {}
        if not args.no_scaling_legs:
            tot = args.channels_total
            for fll in (False, True):
                key = "chain_fll" if fll else "chain"
                strong = bench_chain.run_chain(Q, torch, d, world, rank, stream, use_fll=fll, channels_per_gpu=tot // world,
                                               parity_channels=(256 if world == 1 else 64) if not args.no_cpu else 0,
                                               label=f"strong: {tot} channels in total, {tot // world} per GPU", **common)
                scaling_legs[key + "_strong"] = strong
                if world == 1:
                    scaling_legs[key + "_saturated"] = dict(strong, label=f"saturated weak: {tot} channels per GPU (same run as the strong leg at N = 1)")
                else:
                    scaling_legs[key + "_saturated"] = bench_chain.run_chain(
                        Q, torch, d, world, rank, stream, use_fll=fll, channels_per_gpu=tot, parity_channels=0,
                        label=f"saturated weak: {tot} channels per GPU", **common)
        modulator = bench_chain.run_modulator(Q, torch, d, world, rank, stream, steps=args.steps, warmup=args.warmup,
                                              hbm_peak=hbm_peak, parity=cpu_legs)
        chain_e2e = chain_fll_e2e = modulator_e2e = None
        if not args.no_e2e:
            chain_e2e = bench_chain.run_chain_e2e(Q, torch, d, world, rank, stream, steps=args.steps, use_fll=False)
            chain_fll_e2e = bench_chain.run_chain_e2e(Q, torch, d, world, rank, stream, steps=args.steps, use_fll=True)
            modulator_e2e = bench_chain.run_modulator_e2e(Q, torch, d, world, rank, steps=args.steps)
        stream_leg = bench_chain.run_stream(Q) if (rank == 0 and world == 1 and not args.no_cpu) else None

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        cpu = cpu_baseline(23)

    if rank == 0:
        total_samples = world * args.steps * len(filters) * n
        line = {
            "metric": METRIC, "value": total_samples / (ms_max * 1e-3) / 1e6, "unit": "Msamples/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_max / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"fir_sweep: streaming real-tap RRC FIR, taps {{33,65,129,257}}, 2^{args.log2_samples} cf32 samples "
                                   f"per GPU per tap count (BASELINE.json configs[1])",
                       "l2": "inputs 2 GiB + outputs 2 GiB per launch >> 126 MB L2; no flush needed",
                       "parallelism": f"{world} independent streams, one per GPU, no collective"},
            "roofline": roofline, "roofline_hbm": roofline_hbm, "roofline_by_taps": roofs, "fir_parity": fir_parity, "decimate": decimate, "fma_peak_tflops_measured": fma_peak,
            "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": int(launches), "clocks": clk,
            "build_id": build_id, "cpu_affinity": affinity,
            "scaling_note": "`scaling: weak` refers to `value` (one independent 2^28-sample FIR stream per GPU, no communication). "
                            "The chain legs state their own: chain / chain_fll are weak (2048 channels per GPU), *_strong shard a "
                            "fixed 16384-channel set (config 4), *_saturated put 16384 channels on every GPU",
        }
        if comm is not None:
            line["comm"] = dict(comm.info(), api="qpsk_comm_create / qpsk_ber_gather (ncclAllGather behind the C ABI)")
        if chain is not None:
            line["chain"] = chain
            line["chain_fll"] = chain_fll
            line.update(scaling_legs)
            line["modulator"] = modulator
            if chain_e2e is not None:
                chain["e2e"] = chain_e2e
                chain_fll["e2e"] = chain_fll_e2e
                modulator["e2e"] = modulator_e2e
            if stream_leg is not None:
                line["stream"] = stream_leg
    if comm is not None:
        comm.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank == 0:
        sys.stdout.flush()
        print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
