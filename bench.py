#!/usr/bin/env python
"""bench.py -- headline benchmark of the uplink OFDM receiver hot path on B200.

    python bench.py --gpus N --steps K --warmup W [--impl ours|reference] [--config c2] [--dump-outputs DIR]

Metric (BASELINE.json): LS+MRC antenna-samples/s.  One antenna-sample = one complex64 time
sample from one antenna, cyclic prefix included (A*S*(N+C) per frame).  A "step" is one pass
of the whole hot path (pilot kernel + data kernel) over one batch of F synthetic frames per
GPU.  Default workload: configs[1] = c2 (1024-pt FFT, 64 antennas, 1 pilot + 100 data
symbols, 16-QAM); the 10k-frame batch (563 GB) does not fit HBM, so it is processed in
resident chunks of F frames -- one chunk = one step (weak scaling: F frames per GPU per step).

Printed JSON line (rank 0): value = whole-job antenna-samples/s with inputs resident in HBM;
e2e = the same metric through the public host-buffer call (lsmrc_demod_frames_host: pinned host
buffers, H2D and D2H inside the timed region); roofline = algorithmic HBM bytes of the dominant
(data) kernel / its CUDA-event duration vs the measured copy bandwidth; cpu_baseline = the CPU
oracle (port of the reference's cpuLS path) timed on this box's host cores on a bounded sample.

--impl reference times the reference's CPU path (the oracle port, all host threads) on the
same config and prints the same line with "impl": "reference".
"""
from __future__ import annotations

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

METRIC = "ls_mrc_antenna_samples_per_s"
UNIT = "antenna-samples/s"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=40, help="timed steps; 40 x 256 frames = the 10k-frame batch of config c2")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="c2")
    ap.add_argument("--frames", type=int, default=0, help="frames per step per GPU (0 = config default)")
    ap.add_argument("--e2e-frames", type=int, default=0, help="frames per e2e step per GPU (0 = default)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the c5 latency and other-config legs")
    ap.add_argument("--no-scaling-c4", action="store_true", help="skip the config-4 block that every rank runs")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed (seeded sample of frames) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    return args


# frames per step per GPU: large enough that one step's input exceeds the 126 MB L2 many times over
DEFAULT_FRAMES = {"c1": 65536, "c2": 256, "c3": 192, "c4": 48, "c5": 16384}
DEFAULT_E2E_FRAMES = {"c1": 16384, "c2": 16, "c3": 32, "c4": 8, "c5": 8192}


def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


class ClockSampler:
    """nvidia-smi clocks/throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
                pw.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        # median over the samples taken under load (power well above idle)
        loaded = [s for s, p in zip(sm, pw) if p > 0.6 * max(pw)] if pw else sm
        return {"sm_mhz": statistics.median(loaded) if loaded else None,
                "sm_max_mhz": max(mx) if mx else None, "power_w_max": max(pw) if pw else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def profile_traffic_per_frame(cfg_name):
    """dram bytes per frame of the data kernel from the committed ncu capture, if any"""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p)).get(cfg_name)
            if d:
                return float(d["data_kernel_dram_bytes"]) / float(d["frames"])
        except Exception:
            pass
    return None


def pin_to_gpu_numa(local):
    """Run this rank on the cores of the NUMA node its GPU hangs off (first-touch then places the pinned staging
    buffers there too).  Returns a short description for the JSON line."""
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(local), "--query-gpu=pci.bus_id", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=10).stdout.strip()
        bdf = out.lower().replace("00000000:", "0000:")
        base = "/sys/bus/pci/devices/" + bdf
        node = open(base + "/numa_node").read().strip()
        cpus = open(base + "/local_cpulist").read().strip()
        ids = set()
        for part in cpus.split(","):
            lo, _, hi = part.partition("-")
            ids.update(range(int(lo), int(hi or lo) + 1))
        allowed = os.sched_getaffinity(0)
        use = (ids & allowed) or allowed
        os.sched_setaffinity(0, use)
        return {"gpu_pci": bdf, "numa_node": int(node), "cpus": cpus, "pinned_to": len(use)}
    except Exception as e:  # affinity is an optimisation, never a failure
        return {"error": str(e)[:120]}


def cpu_strong_baseline(cfg, budget_s=8.0):
    """'Strong CPU' comparator promised in BASELINE.md: the same chain (CP strip, FFT, LS, MRC, hard demap left out)
    as a vectorised torch pipeline on all host cores -- torch.fft on CPU is MKL/pocketfft, multi-threaded.  It is NOT
    the reference's code (that is cpu_baseline / --impl reference); it answers 'what would a tuned CPU library do'."""
    import numpy as np
    import torch

    import ofdm_b200 as m

    A, N, C, S, K = cfg.n_ant, cfg.fft_size, cfg.cp_len, cfg.n_sym, cfg.K
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    F = max(1, min(8, int(1.5e9 // cfg.rx_bytes_per_frame)))
    g = torch.Generator().manual_seed(5)
    rx = torch.view_as_complex(torch.randn((F, S, A, N + C, 2), generator=g))
    xb = torch.from_numpy(m.synth.asc_to_bin(m.synth.make_pilot(K, cfg.seed)))

    def run():
        y = torch.fft.fft(rx[..., C:], dim=-1)[..., 1:]           # [F,S,A,K], DC dropped
        h = y[:, 0] / xb                                           # LS estimate [F,A,K]
        e = (h.real ** 2 + h.imag ** 2).sum(1)                     # sum_a |H|^2 [F,K]
        out = (y[:, 1:] * h.conj()[:, None]).sum(2) / e[:, None]   # MRC [F,S-1,K]
        return torch.roll(out, (K + 1) // 2, dims=-1)              # ascending frequency

    run()
    t0 = time.perf_counter()
    reps = 0
    while True:
        run()
        reps += 1
        if time.perf_counter() - t0 > budget_s or reps >= 200:
            break
    dt = time.perf_counter() - t0
    return {"value": reps * F * cfg.antenna_samples_per_frame / dt, "unit": UNIT, "cores": cores, "kind": "torch-cpu",
            "sample": f"{reps} passes over {F} frames of {cfg.name} ({dt:.1f} s): torch.fft.fft + vectorised LS/MRC on {cores} threads "
                      f"(torch {torch.__version__}); not the reference's code, no demapper"}


def h2d_ceiling(dev, nbytes, dist, world, reps=10):
    """What the box's PCIe / host memory delivers to N GPUs at once: every rank copies `nbytes` from a pinned buffer
    with plain cudaMemcpyAsync (three copies in flight), barrier both sides, max over ranks."""
    import torch

    n = max(1, nbytes // 3)
    src = [torch.empty(n, dtype=torch.uint8).pin_memory() for _ in range(3)]
    for b in src:
        b.fill_(1)  # first touch on this rank's NUMA node
    dst = [torch.empty(n, dtype=torch.uint8, device=dev) for _ in range(3)]
    streams = [torch.cuda.Stream(dev) for _ in range(3)]

    def once():
        for i in range(3):
            with torch.cuda.stream(streams[i]):
                dst[i].copy_(src[i], non_blocking=True)

    once()
    torch.cuda.synchronize(dev)
    best = 0.0
    for _ in range(3):  # a ceiling: the best of three trials (a single trial is now and then 5 % low)
        if dist is not None:
            dist.barrier()
        t0 = time.perf_counter()
        for _ in range(reps):
            once()
        torch.cuda.synchronize(dev)
        dt = time.perf_counter() - t0
        t = torch.tensor([dt], device=dev, dtype=torch.float64)
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        best = max(best, world * 3 * n * reps / float(t.item()) / 1e9)
    return best


def scaling_c4_leg(m, dev, local, rank, world, dist, peak, frames=512, steps=5, warmup=2, unique=64):
    """BASELINE config 4 -- the named scaling run: 4096-pt FFT, 256 antennas, 64-QAM, 512 frames per GPU (weak scaling,
    64 GB of antenna samples resident per GPU), every rank on its own frames, no collective on the path.  Runs on ALL
    ranks of every --gpus N line; time = max over ranks."""
    import numpy as np
    import torch

    cfg = m.CONFIGS["c4"]
    free_b, _ = torch.cuda.mem_get_info(dev)
    frames = int(min(frames, max(unique, (free_b * 0.8) // cfg.rx_bytes_per_frame)))
    uniq = min(unique, frames)
    rx_u, pilot_asc, src = m.synth.make_frames_torch(uniq, cfg, dev, seed=cfg.seed + 1000 * rank, chunk=4)
    rx = torch.empty((frames, cfg.n_sym, cfg.n_ant, cfg.fft_size + cfg.cp_len), dtype=torch.complex64, device=dev)
    for f0 in range(0, frames, uniq):   # distinct frames generated once, repeated to fill the batch
        nf = min(uniq, frames - f0)
        rx[f0:f0 + nf] = rx_u[:nf]
    del rx_u
    rx_f = torch.view_as_real(rx)
    comb = torch.empty((frames, cfg.n_sym - 1, cfg.K, 2), device=dev, dtype=torch.float32)
    bits = torch.empty((frames, cfg.n_sym - 1, cfg.bits_row_bytes), device=dev, dtype=torch.uint8)
    stream = torch.cuda.current_stream(dev)
    assert stream.cuda_stream != 0, "the bench runs on its own non-default stream"
    with m.LsMrcReceiver.from_config(cfg, device=local) as r:
        r.set_pilot(pilot_asc)
        r.set_stream(stream.cuda_stream)
        for _ in range(warmup):
            r.demod_frames_device(rx_f, frames, comb, bits)
        torch.cuda.synchronize(dev)
        if dist is not None:
            dist.barrier()
        r.set_timing(True)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(steps):
            r.demod_frames_device(rx_f, frames, comb, bits)
        e1.record(stream)
        torch.cuda.synchronize(dev)
        if dist is not None:
            dist.barrier()
        ms = e0.elapsed_time(e1)
        p_ms, d_ms = r.kernel_ms_history(steps)
        plan = r.describe_plan()
        n_one = r.one_launch_frames_count()
        r.set_stream(None)
    # every decoded frame against the transmitted bits (the repeated frames against the source of their original)
    want = torch.from_numpy(m.synth.pack_bits_rows(src.cpu().numpy(), cfg.qam_bits)).to(dev)
    errs = 0
    for f0 in range(0, frames, uniq):
        nf = min(uniq, frames - f0)
        x = bits[f0:f0 + nf] ^ want[:nf]
        errs += int((x != 0).sum().item())      # bytes that differ
    t = torch.tensor([ms, float(errs)], device=dev, dtype=torch.float64)
    tmax = t.clone()
    if dist is not None:
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
    ms_max = float(tmax[0].item())
    per_gpu_gbs = frames * steps * cfg.algorithmic_bytes_per_frame / (ms_max * 1e-3) / 1e9
    gather = None
    if dist is not None:
        # the one optional exchange of the path (SURVEY 8e): decoded bits of every rank to rank 0 over NCCL, after and
        # outside the timed region; checked by a checksum of checksums (every rank's byte sum travels separately)
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        m.sharding.gather_rows(bits[:1].contiguous(), world)        # communicator warm-up
        torch.cuda.synchronize(dev)
        dist.barrier()
        g0.record(stream)
        everything = m.sharding.gather_rows(bits, frames * world)
        g1.record(stream)
        torch.cuda.synchronize(dev)
        sums = torch.zeros(world, device=dev, dtype=torch.int64)
        sums[rank] = bits.sum(dtype=torch.int64)
        dist.all_reduce(sums, op=dist.ReduceOp.SUM)
        ok = None
        if rank == 0:
            got = everything.view(world, -1).sum(dim=1, dtype=torch.int64)
            ok = bool(torch.equal(got, sums)) and bool(torch.equal(everything[:frames], bits))
        gather = {"backend": dist.get_backend(), "to_rank": 0, "bytes_per_gpu": int(bits.numel()), "ms": g0.elapsed_time(g1),
                  "share_of_step": g0.elapsed_time(g1) / (ms_max / steps), "checksums_match": ok,
                  "what": "sharding.gather_rows of the packed bits of all ranks, after the timed region"}
        del everything
    del rx, rx_f, comb, bits, want
    torch.cuda.empty_cache()
    return {"workload": "c4: 4096-pt FFT, CP 288, 256 antennas, 1 pilot + 13 data symbols, 64-QAM", "scaling": "weak",
            "frames_per_gpu": frames, "distinct_frames_per_gpu": uniq, "steps": steps, "warmup": warmup,
            "input_bytes_per_gpu": frames * cfg.rx_bytes_per_frame, "ms_per_step": ms_max / steps,
            "value": world * frames * steps * cfg.antenna_samples_per_frame / (ms_max * 1e-3), "unit": UNIT,
            "algorithmic_gbs_per_gpu": per_gpu_gbs, "frac_of_hbm_peak": per_gpu_gbs / peak,
            "pilot_kernel_ms": statistics.mean(p_ms), "data_kernel_ms": statistics.mean(d_ms),
            "kernels": "one persistent launch (pilot items, then data items): the whole step is data_kernel_ms" if n_one > 0
                       else "pilot kernel + data kernel",
            "differing_bit_bytes_vs_source_all_ranks": int(t[1].item()) if dist is not None else errs,
            "frames_checked_per_gpu": frames, "plan": plan, "bits_gather": gather}


def cpu_baseline(cfg, n_threads, budget_s=12.0):
    """oracle port (restated cpuLS.hpp path + demap) timed on the host cores, bounded sample"""
    import numpy as np
    from oracle import oracle_py

    oracle_py.build(ref=False)
    import ofdm_b200 as m

    rng = np.random.default_rng(7)
    A, N, C, S = cfg.n_ant, cfg.fft_size, cfg.cp_len, cfg.n_sym
    pilot = m.synth.make_pilot(cfg.K, cfg.seed)

    def make(F):
        x = rng.standard_normal((F, S, A, N + C, 2), dtype=np.float32)
        return x.view(np.complex64)[..., 0]

    # calibrate on one frame per thread
    F0 = n_threads
    rx = make(F0)
    t0 = time.perf_counter()
    oracle_py.demod_frames(rx, pilot, cfg.qam_bits, C, n_threads=n_threads, fast=True)
    t_cal = time.perf_counter() - t0
    reps = max(1, min(int(budget_s / max(t_cal, 1e-3)), 2000))
    t0 = time.perf_counter()
    for _ in range(reps):
        oracle_py.demod_frames(rx, pilot, cfg.qam_bits, C, n_threads=n_threads, fast=True)
    dt = time.perf_counter() - t0
    frames = F0 * reps
    ref1 = None
    if oracle_py.ref_binary(A, N, C, S) is not None:  # the reference's own build, as --impl reference times it
        fr, secs = oracle_py.time_reference(make(2), pilot, C)
        ref1 = {"value": fr * cfg.antenna_samples_per_frame / secs, "unit": UNIT, "cores": 1, "kind": "reference",
                "sample": f"{fr} frames through oracle/_ref (reference cpuLS.hpp + ring + file output), {secs:.2f} s"}
    return {"reference_1core": ref1,
            "value": frames * cfg.antenna_samples_per_frame / dt, "unit": UNIT, "cores": n_threads, "kind": "port",
            "sample": f"{frames} frames of {cfg.name} ({F0} frames x {reps} passes, {dt:.1f} s), oracle/cpuls_oracle.c "
                      f"-O3 -march=native, FFT = oracle/fft_shim.c (FFTW3 absent), frames split over {n_threads} threads"}


def run_reference(args, cfg):
    """--impl reference: the reference's own CPU implementation of the path, same metric and config.
    When oracle/_ref holds a build of the reference's cpuLS.hpp for these dimensions (compiled from
    /root/reference by oracle/Makefile; FFT through the shim because FFTW3 is absent) that binary is timed:
    one process, one thread -- the reference is single-threaded and its ring name is hard-coded.  Otherwise
    the oracle port runs with all host threads."""
    rank, world, _ = dist_env()
    if rank != 0:
        return
    import numpy as np
    from oracle import oracle_py
    import ofdm_b200 as m

    A, N, C, S = cfg.n_ant, cfg.fft_size, cfg.cp_len, cfg.n_sym
    pilot = m.synth.make_pilot(cfg.K, cfg.seed)
    rng = np.random.default_rng(11)

    def frames(F):
        return rng.standard_normal((F, S, A, N + C, 2), dtype=np.float32).view(np.complex64)[..., 0]

    if oracle_py.ref_binary(A, N, C, S) is not None:
        kind, cores = "reference", 1
        _, t1 = oracle_py.time_reference(frames(1), pilot, C)        # calibration, also warms the page cache
        F = int(max(1, min(4, 100.0 / max(args.steps + args.warmup, 1) / max(t1, 1e-3))))
        rx = frames(F)
        for _ in range(args.warmup):
            oracle_py.time_reference(rx, pilot, C)
        dt = 0.0
        for _ in range(args.steps):
            dt += oracle_py.time_reference(rx, pilot, C)[1]
        sample = (f"{F} frames of {cfg.name} per step through oracle/_ref/cpuls_ref_{oracle_py.ref_case_name(A, N, C, S)}: the "
                  f"reference's cpuLS.hpp + ring + Output_cpu.dat path, 1 thread, FFT = oracle/fft_shim.c (FFTW3 absent)")
    else:
        oracle_py.build(ref=False)
        kind, cores = "port", os.cpu_count() or 1
        F = max(1, min(cores, max(1, int(2e9 // cfg.rx_bytes_per_frame))))
        rx = frames(F)
        for _ in range(args.warmup):
            oracle_py.demod_frames(rx, pilot, cfg.qam_bits, C, n_threads=cores, fast=True)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            oracle_py.demod_frames(rx, pilot, cfg.qam_bits, C, n_threads=cores, fast=True)
        dt = time.perf_counter() - t0
        sample = (f"{F} frames of {cfg.name} per step on {cores} host threads; oracle port of cpuLS.hpp "
                  f"(no reference build for these dimensions in oracle/_ref)")
    value = args.steps * F * cfg.antenna_samples_per_frame / dt
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(cfg, F, None),
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def latency_leg(m, dev_index, n_launch=10000):
    """BASELINE config c5: one frame per call (64-pt FFT, 16 antennas, 16 symbols, QPSK), 10,000 calls,
    p50/p99 per-frame latency.  Measured by host/latency_main (C++, steady_clock around the C-ABI calls, no
    Python in the loop): device-resident frame (`lsmrc_demod_frames_device` + `lsmrc_sync`) and pinned host
    frame with results back on the host (`lsmrc_demod_frames_host`), under the default launch policy (ONE fused
    kernel per frame; host buffers read and written in place) and with the pilot + data kernel pair; the
    `floor_trivial_kernel` entry is the same call pattern around a one-row copy kernel."""
    cfg = m.CONFIGS["c5"]
    host = os.path.join(ROOT, "gpu-accel-ofdm-ls-mrc_b200", "host")
    if subprocess.run(["make", "-C", host, "--no-print-directory"], capture_output=True).returncode != 0:
        return {"error": "host programs did not build"}
    env = dict(os.environ, CUDA_VISIBLE_DEVICES=os.environ.get("CUDA_VISIBLE_DEVICES", str(dev_index)))
    r = subprocess.run([os.path.join(host, "bin", "latency_main"), "--rows", str(cfg.n_ant), "--cols", str(cfg.fft_size),
                        "--prefix", str(cfg.cp_len), "--syms", str(cfg.n_sym), "--qam", str(cfg.qam_bits),
                        "--launches", str(n_launch)], capture_output=True, text=True, timeout=300, env=env)
    if r.returncode != 0:
        return {"error": (r.stdout + r.stderr)[-300:]}
    res = json.loads(r.stdout.strip().splitlines()[-1])
    out = {"workload": "c5: 64-pt FFT, 16 antennas, 16 symbols, QPSK, one frame per call", "launches": n_launch}
    out.update(res["device_one_launch"])           # headline: p50_us / p99_us / mean_us of the device-resident call
    out["host_buffers_in_place"] = res["host_one_launch_in_place"]
    out["host_buffers_staged_copies"] = res["host_one_launch_staged"]
    out["two_kernel_path"] = {"device": res["device_two_kernels"], "host_buffers": res["host_two_kernels"]}
    out["floor_trivial_kernel"] = res["floor_trivial_kernel"]
    out["what"] = ("C++ steady_clock around the C-ABI call(s) per frame; p50_us/p99_us = device-resident frame, one fused "
                   "kernel + sync; host_buffers_* = pinned host frame in, results on the host out")
    return out


def other_configs_leg(m, dev_index, peak):
    """kernel-time throughput of the remaining BASELINE dimension sets (parity for them is in tests/)"""
    import torch

    out = {}
    dev = torch.device("cuda", dev_index)
    for name, frames in (("c1", 16384), ("c3", 384), ("c4", 192)):
        cfg = m.CONFIGS[name]
        rx = torch.randn((frames, cfg.n_sym, cfg.n_ant, cfg.fft_size + cfg.cp_len, 2), device=dev)
        comb = torch.empty((frames, cfg.n_sym - 1, cfg.K, 2), device=dev)
        bits = torch.empty((frames, cfg.n_sym - 1, cfg.bits_row_bytes), device=dev, dtype=torch.uint8)
        with m.LsMrcReceiver.from_config(cfg, device=dev_index) as r:
            r.set_pilot(m.synth.make_pilot(cfg.K, 1))
            r.set_timing(True)
            ms = []
            for _ in range(6):
                r.demod_frames_device(rx, frames, comb, bits)
                a, b = r.last_kernel_ms()
                ms.append(a + b)
            t = statistics.median(ms[2:])
            gbs = frames * cfg.algorithmic_bytes_per_frame / (t * 1e-3) / 1e9
            out[name] = {"frames": frames, "ms": t, "antenna_samples_per_s": frames * cfg.antenna_samples_per_frame / (t * 1e-3),
                         "algorithmic_gbs": gbs, "frac_of_hbm_peak": gbs / peak, "plan": r.describe_plan()}
        del rx, comb, bits
        torch.cuda.empty_cache()
    return out


def frontend_leg(m, dev_index, peak):
    """the front end that precedes the hot path (rx_and_corr.cpp:332-393) on the GPU: PN frame sync over a whole
    c2-sized capture and the stitching of the frame into the receiver's input layout"""
    import torch

    cfg = m.CONFIGS["c2"]
    dev = torch.device("cuda", dev_index)
    L = 255
    samps = L + cfg.n_sym * (cfg.fft_size + cfg.cp_len) + 512
    b1 = 0.05 * torch.randn((cfg.n_ant, samps, 2), device=dev)
    b2 = 0.05 * torch.randn((cfg.n_ant, samps, 2), device=dev)
    pn = torch.view_as_real(torch.from_numpy(m.synth.make_pn()).to(dev)).contiguous()
    b1[:, 300:300 + L, 0] = pn[:, 0]
    b1[:, 300:300 + L, 1] = 0
    rx = torch.empty((cfg.n_sym, cfg.n_ant, cfg.fft_size + cfg.cp_len, 2), device=dev)
    with m.LsMrcReceiver.from_config(cfg, device=dev_index) as r:
        stream = torch.cuda.current_stream(dev)
        assert stream.cuda_stream != 0, "the bench runs on its own non-default stream"
        r.set_stream(stream.cuda_stream)
        for _ in range(3):
            off = r.sync_correlate(b1, cfg.n_ant, samps, pn, L, 0.5)[0]
            r.sync_assemble(b1, b2, samps, max(off, 0), L, rx)
        e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
        e[0].record(stream)
        for _ in range(10):
            off = r.sync_correlate(b1, cfg.n_ant, samps, pn, L, 0.5)[0]
        e[1].record(stream)
        for _ in range(10):
            r.sync_assemble(b1, b2, samps, off, L, rx)
        e[2].record(stream)
        torch.cuda.synchronize(dev)
    t_corr, t_asm = e[0].elapsed_time(e[1]) / 10, e[1].elapsed_time(e[2]) / 10
    taps = cfg.n_ant * (samps - L + 1) * L
    return {"workload": f"c2 capture: {cfg.n_ant} channels x {samps} samples, PN 255", "offset_found": off,
            "correlate_ms": t_corr, "correlate_gmac_per_s": taps / (t_corr * 1e-3) / 1e9,
            "assemble_ms": t_asm, "assemble_gbs": 2 * rx.numel() * 4 / (t_asm * 1e-3) / 1e9,
            "assemble_frac_of_hbm_peak": 2 * rx.numel() * 4 / (t_asm * 1e-3) / 1e9 / peak}


def ring_stream_leg(m, n_frames=768, feeder_threads=None, config="c3", lanes=3, note=None, batch=1, feeder_args=()):
    """BASELINE config c3: 14-symbol slots of a 2048-pt / 128-antenna system streamed through the pinned
    shared-memory ring (producer process = host/ring_feeder, consumer = host/stream_main: whole frames DMA'd
    out of the ring on 3 rotating lanes, H2D of frame i+1 overlapping the kernels of frame i)."""
    import shutil
    import tempfile
    import uuid

    import numpy as np

    cfg = m.CONFIGS[config]
    if feeder_threads is None:
        # measured on a 16-core host, one slot in flight per thread: 4 -> 36, 8 -> 54, 12 -> 51, 16 -> 48 GB/s of slots
        feeder_threads = max(1, min(8, (os.cpu_count() or 2) - 4))
    host = os.path.join(ROOT, "gpu-accel-ofdm-ls-mrc_b200", "host")
    if subprocess.run(["make", "-C", host, "--no-print-directory"], capture_output=True).returncode != 0:
        return {"error": "host programs did not build"}
    d = tempfile.mkdtemp(prefix="lsmrc_ring_", dir="/dev/shm" if os.path.isdir("/dev/shm") else None)
    try:
        base = 8  # distinct frames on disk; the feeder loops over them
        rng = np.random.default_rng(3)
        rx = rng.standard_normal((base, cfg.n_sym, cfg.n_ant, cfg.fft_size + cfg.cp_len, 2), dtype=np.float32)
        rx.tofile(os.path.join(d, "rx.bin"))
        m.synth.make_pilot(cfg.K, cfg.seed).tofile(os.path.join(d, "Pilots.dat"))
        shm = "/lsmrc_" + uuid.uuid4().hex[:8]
        ring = (lanes * batch + 1) * cfg.n_sym + 1
        dims = ["--rows", str(cfg.n_ant), "--cols", str(cfg.fft_size), "--prefix", str(cfg.cp_len), "--syms", str(cfg.n_sym),
                "--ring", str(ring), "--shm", shm]
        feeder = subprocess.Popen([os.path.join(host, "bin", "ring_feeder"), "--file", os.path.join(d, "rx.bin"), "--frames", str(base),
                                   "--repeat", str(n_frames // base), "--threads", str(feeder_threads)] + list(feeder_args) + dims)
        try:
            r = subprocess.run([os.path.join(host, "bin", "stream_main"), "--qam", str(cfg.qam_bits), "--frames", str(n_frames),
                                "--pilots", os.path.join(d, "Pilots.dat"), "--no-output", "--lanes", str(lanes), "--batch", str(batch),
                                "--trace", os.path.join(d, "trace.csv")] + dims,
                               cwd=d, capture_output=True, text=True, timeout=300)
            feeder.wait(timeout=60)
        finally:
            if feeder.poll() is None:
                feeder.kill()
            if os.path.exists("/dev/shm" + shm):
                os.unlink("/dev/shm" + shm)
        if r.returncode != 0:
            return {"error": (r.stdout + r.stderr)[-300:]}
        out = json.loads(r.stdout.strip().splitlines()[-1])
        ts = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "trace_summary.py"), os.path.join(d, "trace.csv")],
                            capture_output=True, text=True)
        out["overlap"] = ts.stdout.strip().splitlines() if ts.returncode == 0 else None
        # stream_main counts whole slots (prefix included) as h2d_gbs; what crosses the link is less when the copy leaves the
        # prefix in the ring
        # (frames of at most 512 KiB are read in place by the one-launch kernel: no copy at all)
        stripped = "h2d=strip-cp" in out.get("plan", "") and cfg.rx_bytes_per_frame > (512 << 10)
        out["ingest_gbs"] = out["h2d_gbs"]
        out["link_gbs"] = out["h2d_gbs"] * (cfg.fft_size / (cfg.fft_size + cfg.cp_len) if stripped else 1.0)
        out["workload"] = (f"{config}: {cfg.fft_size}-pt FFT, {cfg.n_ant} antennas, {cfg.n_sym}-symbol slots, ring of {ring} slots "
                           f"({cfg.rx_bytes_per_frame / 1e6:.1f} MB per frame), one producer process filling slots with {feeder_threads} threads")
        out["note"] = note or ("PCIe-bound: the H2D engine is busy 98 % of the time; the consumer overlaps H2D, both kernels and D2H on "
                               "3 lanes (a producer that only publishes slots: 57.8 GB/s of slots on the same box)")
        return out
    finally:
        shutil.rmtree(d, ignore_errors=True)


def dump_outputs(out_dir, comb, bits, budget=48 << 20):
    """What the timed call hands its caller, for a fixed, seeded sample of the batch's frames (at most `budget`
    bytes), so that two builds can be compared output for output on the same inputs.  float32 .npy files:
    combined [n, S-1, K, 2] (re, im), bits [n, S-1, row bytes] (the packed bytes, values 0..255), and
    frames [n] (float64), the sampled frame indices."""
    import numpy as np
    import torch

    F = comb.shape[0]
    n = max(1, min(F, budget // (4 * (comb[0].numel() + bits[0].numel()))))
    idx = np.sort(np.random.default_rng(0).choice(F, size=n, replace=False))
    sel = torch.from_numpy(idx).to(comb.device)
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "combined.npy"), comb.index_select(0, sel).cpu().numpy())
    np.save(os.path.join(out_dir, "bits.npy"), bits.index_select(0, sel).cpu().numpy().astype(np.float32))
    np.save(os.path.join(out_dir, "frames.npy"), idx.astype(np.float64))


def workload_config(cfg, frames, e2e_frames):
    return {"workload": f"{cfg.name}: {cfg.fft_size}-pt FFT, CP {cfg.cp_len}, {cfg.n_ant} antennas, 1 pilot + "
                        f"{cfg.n_sym - 1} data symbols, {1 << cfg.qam_bits}-QAM",
            "frames_per_step_per_gpu": frames, "e2e_frames_per_step_per_gpu": e2e_frames,
            "input_bytes_per_step_per_gpu": frames * cfg.rx_bytes_per_frame,
            "l2_policy": "inputs larger than L2 (each step streams its whole batch from HBM once)",
            "note": "10k-frame batch processed as resident chunks; one chunk = one step"}


def main():
    args = parse_args()
    import ofdm_b200 as m

    cfg = m.CONFIGS[args.config]
    if args.impl == "reference":
        run_reference(args, cfg)
        return

    import numpy as np
    import torch

    rank, world, local = dist_env()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the receiver has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    affinity = pin_to_gpu_numa(local)
    dist = None
    if world > 1:
        import torch.distributed as dist_mod

        dist = dist_mod
        dist.init_process_group("nccl", device_id=dev)

    # a stream of our own, made torch's current one before anything is enqueued (torch's default stream has handle 0,
    # which lsmrc_set_stream reads as "back to the handle's own stream"): the synthetic-data generator, the torch
    # events and the library's launches all share it
    stream = torch.cuda.Stream(dev)
    torch.cuda.set_stream(stream)

    F = args.frames or DEFAULT_FRAMES[cfg.name]
    Fe = args.e2e_frames or DEFAULT_E2E_FRAMES[cfg.name]
    # frames are independent: rank r owns global frames [r*F, (r+1)*F) of every step (no collective on the path)
    rx, pilot_asc, src = m.synth.make_frames_torch(F, cfg, dev, seed=cfg.seed + 1000 * rank, chunk=8)
    rx_f = torch.view_as_real(rx)
    comb = torch.empty((F, cfg.n_sym - 1, cfg.K, 2), device=dev, dtype=torch.float32)
    bits = torch.empty((F, cfg.n_sym - 1, cfg.bits_row_bytes), device=dev, dtype=torch.uint8)
    # host-path chunks of ~450 MB (8 frames of c2): large enough to run the copy engine flat out, three in flight
    chunk_frames = max(1, min(Fe, int(round(450e6 / cfg.rx_bytes_per_frame)) or 1))
    rcv = m.LsMrcReceiver.from_config(cfg, max_frames=chunk_frames, device=local, n_lanes=3)
    rcv.set_pilot(pilot_asc)
    rcv.set_stream(stream.cuda_stream)

    def step():
        rcv.demod_frames_device(rx_f, F, comb, bits)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize(dev)

    # ---- correctness gate on this very batch: decoded bits vs the transmitted bits
    step()
    torch.cuda.synchronize(dev)
    want = torch.from_numpy(m.synth.pack_bits_rows(src[:2].cpu().numpy(), cfg.qam_bits))
    got = bits[:2].cpu()
    bit_errors = int(np.unpackbits((got ^ want).numpy()).sum())
    ber = bit_errors / float(want.numel() * 8)

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()  # samples through warm-up and the timed region; idle samples are filtered by power
    for _ in range(args.warmup):
        step()
    barrier()
    l0 = rcv.launch_count()
    rcv.set_timing(True)  # per-kernel CUDA events on the launching stream, read back after the region
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(stream)
    for _ in range(args.steps):
        step()
    ev1.record(stream)
    barrier()
    ms = ev0.elapsed_time(ev1)
    launches = rcv.launch_count() - l0
    p_ms, d_ms = rcv.kernel_ms_history(min(args.steps, 256))
    rcv.set_timing(False)
    clocks = sampler.stop() if rank == 0 else None
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, comb, bits)
    t = torch.tensor([ms], device=dev, dtype=torch.float64)
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = float(t.item())
    value = world * F * args.steps * cfg.antenna_samples_per_frame / (ms_max * 1e-3)

    # ---- dominant (data) kernel: its CUDA-event durations inside the timed region above
    data_ms = statistics.mean(d_ms)
    pilot_ms = statistics.mean(p_ms)
    A, N, S, K = cfg.n_ant, cfg.fft_size, cfg.n_sym, cfg.K
    data_bytes_per_frame = 8 * A * (S - 1) * N + 8 * (S - 1) * K + (S - 1) * cfg.bits_row_bytes
    peak, peak_src = measured_peak_gbs()
    achieved = F * data_bytes_per_frame / (data_ms * 1e-3) / 1e9
    tpf = profile_traffic_per_frame(cfg.name)
    roofline = {"bound": "hbm", "kernel": ("lsmrc_data_sh" if cfg.fft_size >= 2048 else "lsmrc_kernel<MODE_DATA>") + " (FFT + MRC + demap)",
                "achieved": achieved,
                "peak": peak, "unit": "GB/s", "frac": achieved / peak, "peak_source": peak_src,
                "traffic": (tpf * F) if tpf else None, "algorithmic_bytes_per_launch": F * data_bytes_per_frame,
                "kernel_ms": data_ms, "pilot_kernel_ms": pilot_ms, "kernel_share_of_step": data_ms / (data_ms + pilot_ms),
                "whole_path_achieved": F * cfg.algorithmic_bytes_per_frame / ((data_ms + pilot_ms) * 1e-3) / 1e9}

    # ---- e2e: host buffers through the public call, H2D + D2H inside the timed region
    e2e = None
    if not args.no_e2e:
        h_rx = rcv.pinned_array((Fe, cfg.n_sym, cfg.n_ant, cfg.fft_size + cfg.cp_len), np.complex64)
        h_rx[...] = rx[:Fe].cpu().numpy() if Fe <= F else np.resize(rx.cpu().numpy(), h_rx.shape)
        h_comb = rcv.pinned_array((Fe, cfg.n_sym - 1, cfg.K), np.complex64)
        h_bits = rcv.pinned_array((Fe, cfg.n_sym - 1, cfg.bits_row_bytes), np.uint8)
        n_e2e = max(3, min(args.steps, 10))
        for _ in range(4):  # lanes, staging buffers and the pinned mappings are all touched before timing
            rcv.demod_frames_host(h_rx, Fe, h_comb, h_bits)
        barrier()
        t0 = time.perf_counter()
        for _ in range(n_e2e):
            rcv.demod_frames_host(h_rx, Fe, h_comb, h_bits)
        dt = time.perf_counter() - t0
        t = torch.tensor([dt], device=dev, dtype=torch.float64)
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dt = float(t.item())
        e2e_err = int(np.unpackbits(h_bits[:1] ^ got[:1].numpy()).sum()) if Fe >= 1 else 0
        # the host path leaves the cyclic prefix behind (strided H2D copy): count the bytes actually moved
        strip = "h2d=strip-cp" in rcv.describe_plan()
        h2d = int(h_rx.nbytes * cfg.fft_size // (cfg.fft_size + cfg.cp_len)) if strip else int(h_rx.nbytes)
        ceiling = h2d_ceiling(dev, h2d, dist, world)
        e2e = {"value": world * Fe * n_e2e * cfg.antenna_samples_per_frame / dt, "unit": UNIT,
               "h2d_ceiling_gbs": ceiling, "h2d_frac_of_ceiling": (world * h2d * n_e2e / dt / 1e9) / ceiling,
               "h2d_ceiling_what": f"{world} rank(s) copying the same bytes from plain pinned buffers with cudaMemcpyAsync at the same time",
               "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": int(h_comb.nbytes + h_bits.nbytes),
               "steps": n_e2e, "ms_per_step": 1e3 * dt / n_e2e, "api": "lsmrc_demod_frames_host (pinned host buffers, 3 lanes)",
               "h2d_gbs": world * h2d * n_e2e / dt / 1e9, "host_input_bytes_per_step": int(h_rx.nbytes),
               "h2d_copy": "strided, cyclic prefix left on the host" if strip else "whole slots",
               "bit_mismatch_vs_device_path": e2e_err}
        if not args.no_extras:
            # The same frames as the radio puts them on the wire (int16 I/Q; rx_and_corr.cpp:283 has UHD convert them to
            # complex float on the host), converted on the device after the copy: half the PCIe bytes.  A secondary figure --
            # `e2e` above stays the complex-float call the reference's interface has.
            peak_amp = float(np.abs(h_rx.view(np.float32)).max())
            h_iq = rcv.pinned_array(h_rx.shape + (2,), np.int16)
            np.rint(h_rx.view(np.float32).reshape(h_iq.shape) * (8191.0 / peak_amp), out=h_rx.view(np.float32).reshape(h_iq.shape))
            h_iq[...] = h_rx.view(np.float32).reshape(h_iq.shape)      # (h_rx is scratch from here on)
            sc = 1.0 / 32767.0
            h_bits16 = np.empty_like(h_bits)
            for _ in range(3):
                rcv.demod_frames_host_sc16(h_iq, Fe, sc, h_comb, h_bits)
            h_bits16[...] = h_bits
            barrier()
            t0 = time.perf_counter()
            for _ in range(n_e2e):
                rcv.demod_frames_host_sc16(h_iq, Fe, sc, h_comb, h_bits)
            dt16 = time.perf_counter() - t0
            t = torch.tensor([dt16], device=dev, dtype=torch.float64)
            if dist is not None:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt16 = float(t.item())
            # check: the complex-float call on the floats the host conversion gives must decode the same bits
            h_rx.view(np.float32).reshape(h_iq.shape)[...] = h_iq.astype(np.float32) * np.float32(sc)
            rcv.demod_frames_host(h_rx, Fe, h_comb, h_bits)
            h2d16 = h2d // 2
            e2e["wire_format_sc16"] = {
                "value": world * Fe * n_e2e * cfg.antenna_samples_per_frame / dt16, "unit": UNIT, "ms_per_step": 1e3 * dt16 / n_e2e,
                "h2d_bytes_per_step": h2d16, "h2d_gbs": world * h2d16 * n_e2e / dt16 / 1e9,
                "api": "lsmrc_demod_frames_host_sc16 (int16 I/Q in pinned host memory, converted on the device)",
                "bit_mismatch_vs_complex_float_call_on_converted_samples": int(np.unpackbits(h_bits16 ^ h_bits).sum()),
                "note": "not the reference's interface (complex float): what the link carries when the radio's wire format is kept"}

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu = cpu_baseline(cfg, os.cpu_count() or 1)
        cpu["strong"] = cpu_strong_baseline(cfg)
        if e2e is not None:   # the host-buffer figure next to each CPU figure (the 1-core reference build is the weakest)
            e2e["over_cpu_port_all_cores"] = e2e["value"] / cpu["value"]
            e2e["over_cpu_strong_torch"] = e2e["value"] / cpu["strong"]["value"]
            if cpu.get("reference_1core"):
                e2e["over_reference_1core"] = e2e["value"] / cpu["reference_1core"]["value"]

    # ---- long-run behaviour: this kernel is fp32-heavy (about 40 TFLOP/s at full clocks) and reaches the
    # 1000 W board power cap after ~0.15 s of back-to-back steps, after which the SM clock drops; the
    # named workload (a 10k-frame batch = 40 steps) is shorter than that, so both figures are reported
    sustained = None
    if rank == 0 and world == 1 and not args.no_extras:
        n_long = 300
        samp2 = ClockSampler(local)
        samp2.start()
        rcv.set_timing(True)
        for _ in range(n_long):
            step()
        torch.cuda.synchronize(dev)
        pl, dl = rcv.kernel_ms_history(100)
        rcv.set_timing(False)
        ck2 = samp2.stop()
        dms = statistics.mean(dl)
        ach = F * data_bytes_per_frame / (dms * 1e-3) / 1e9
        sustained = {"steps": n_long, "measured_over_last": len(dl), "data_kernel_ms": dms, "achieved": ach, "frac": ach / peak,
                     "value": F * cfg.antenna_samples_per_frame / ((dms + statistics.mean(pl)) * 1e-3), "clocks": ck2}

    # ---- BASELINE config 4 on every rank (the named scaling configuration); c2 stays `value`
    del rx, rx_f, comb, bits
    torch.cuda.empty_cache()
    scaling_c4 = None
    if not args.no_scaling_c4:
        rcv.set_stream(None)
        scaling_c4 = scaling_c4_leg(m, dev, local, rank, world, dist, peak)

    latency = others = frontend = ring_stream = None
    if rank == 0 and world == 1 and not args.no_extras:
        latency = latency_leg(m, local)
        others = other_configs_leg(m, local, peak)
        frontend = frontend_leg(m, local, peak)
        ring_stream = ring_stream_leg(m)
        # BASELINE config c1 through the ring: tiny frames, read in place by the one-launch kernel, 8 in flight
        ring_stream["c1"] = ring_stream_leg(m, n_frames=32768, feeder_threads=1, config="c1", lanes=4, batch=16,
                                            note="launch-latency bound: one fused kernel per frame reads the ring slots in place "
                                                 "(ring wrap and 4-byte slot alignment included); up to 16 waiting frames per launch, 4 launches in flight")

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms_max / args.steps, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": workload_config(cfg, F, Fe), "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e,
                "gpu_launches": launches, "clocks": clocks, "plan": rcv.describe_plan(), "latency": latency,
                "sustained": sustained, "scaling_c4": scaling_c4, "other_configs": others, "frontend": frontend,
                "ring_stream": ring_stream, "affinity": affinity,
                "parity": {"bit_errors_vs_source": bit_errors, "ber": ber, "frames_checked": 2}}
        print(json.dumps(line), flush=True)
    rcv.close()
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
