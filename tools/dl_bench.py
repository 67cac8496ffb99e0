"""Throughput of the multi-user downlink (lsmrc_precode_frames_device): ZF precoding from the uplink estimate, inverse
row FFT and cyclic prefix, on c2-like (A = 64, N = 1024, C = 64) and c4-like (A = 256, N = 4096, C = 288) arrays with
U = 4 and 8 users and Sd = 13 and 100 downlink symbols per frame.

Each batch moves well over twice the 126 MB L2 per call (channel estimates and symbols in, antenna samples out), so the
timed calls stream from and to HBM.  Per call: CUDA events around the call, >= 5 warm-ups, >= 20 timed calls, median.
The library's own phase events (lsmrc_set_timing) split each call into the precoder build (inverse and per-frame gain)
and the precode phase (bin-order layout pass and the fused precode / inverse-FFT / CP kernel).  Algorithmic bytes per
frame: 8*A*Sd*(N+C) written + 8*U*A*N + 8*Sd*U*K read, over the device-to-device copy rate measured in the same run.
One JSON line per case with the card name and power limit read in the same run.

  python tools/dl_bench.py [--quick] [--out DIR]
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

L2_BYTES = 126 << 20

# (name, A, N, C, U, Sd, frames): frames chosen so that every call moves > 2x L2 and gives every SM work
CASES = [
    ("c2", 64, 1024, 64, 4, 13, 64),
    ("c2", 64, 1024, 64, 8, 13, 64),
    ("c2", 64, 1024, 64, 4, 100, 16),
    ("c2", 64, 1024, 64, 8, 100, 16),
    ("c4", 256, 4096, 288, 4, 13, 8),
    ("c4", 256, 4096, 288, 8, 13, 8),
    ("c4", 256, 4096, 288, 4, 100, 4),
    ("c4", 256, 4096, 288, 8, 100, 4),
]


def algorithmic_bytes(A, N, C, U, Sd):
    """per frame: antenna samples out (8*A*Sd*(N+C)) + precoder in (8*U*A*N) + user symbols in (8*Sd*U*K)"""
    return 8 * A * Sd * (N + C) + 8 * U * A * N + 8 * Sd * U * (N - 1)


def card():
    import torch

    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit", "--format=csv,noheader"], capture_output=True,
                            text=True, timeout=30).stdout.strip()
    except Exception as e:  # (reported, not guessed)
        pl = f"unknown ({e.__class__.__name__})"
    return name, pl


def copy_peak_gbps(warmup=3, iters=10, nbytes=2 << 30):
    """device-to-device copy rate (bytes read + written per second) of a buffer far larger than L2"""
    import torch

    src = torch.empty(nbytes // 4, dtype=torch.float32, device="cuda:0")
    dst = torch.empty_like(src)
    src.fill_(1.0)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(warmup):
        dst.copy_(src)
    ts = []
    for _ in range(iters):
        e0.record()
        dst.copy_(src)
        e1.record()
        e1.synchronize()
        ts.append(e0.elapsed_time(e1))
    del src, dst
    torch.cuda.empty_cache()
    return 2 * nbytes / (statistics.median(ts) * 1e-3) / 1e9


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--quick", action="store_true", help="first two cases only, one frame each (rehearsal)")
    ap.add_argument("--out", default=None, help="also append the JSON lines to DIR/dl_bench.jsonl")
    args = ap.parse_args()
    import torch

    import ofdm_b200

    if not torch.cuda.is_available():
        raise SystemExit("dl_bench needs a CUDA GPU")
    dev = torch.device("cuda:0")
    name, power = card()
    peak = copy_peak_gbps()
    lines = []
    for (tag, A, N, C, U, Sd, F) in (CASES[:2] if args.quick else CASES):
        K = N - 1
        per_frame = algorithmic_bytes(A, N, C, U, Sd)
        if args.quick:
            F = 1
        else:
            assert F * per_frame > 2 * L2_BYTES
        g = torch.Generator(device=dev).manual_seed(1)
        hc = torch.randn((F, U, A, K), dtype=torch.complex64, device=dev, generator=g)
        sym = torch.randn((F, Sd, U, K), dtype=torch.complex64, device=dev, generator=g)
        tx = torch.empty((F, Sd, A, N + C), dtype=torch.complex64, device=dev)
        gain = torch.empty((F,), dtype=torch.float32, device=dev)
        torch.cuda.synchronize()
        st = torch.cuda.Stream(dev)  # (a stream of its own: handle 0 would select the receiver's internal stream)
        with ofdm_b200.LsMrcReceiver(A, N, C, 2, 4) as r, torch.cuda.stream(st):
            r.set_stream(st.cuda_stream)

            def call():
                r.precode_frames_device(hc, F, U, sym, Sd, tx, gain)

            for _ in range(args.warmup):
                call()
            st.synchronize()
            r.set_timing(True)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ts = []
            for _ in range(args.iters):
                e0.record(st)
                call()
                e1.record(st)
                e1.synchronize()
                ts.append(e0.elapsed_time(e1))
            build_ms, precode_ms = r.kernel_ms_history(args.iters)
            r.set_timing(False)
            r.set_stream(None)
        t = statistics.median(ts)
        byt = F * per_frame
        rec = {"case": tag, "A": A, "N": N, "C": C, "U": U, "Sd": Sd, "frames": F, "MB_per_call": round(byt / 1e6, 1),
               "ms_call": round(t, 4), "ms_build": round(statistics.median(build_ms), 4),
               "ms_precode": round(statistics.median(precode_ms), 4),
               "alg_GBps": round(byt / (t * 1e-3) / 1e9, 1), "alg_GBps_precode_phase": round(byt / (statistics.median(precode_ms) * 1e-3) / 1e9, 1),
               "copy_peak_GBps": round(peak, 1), "hbm_fraction": round(byt / (t * 1e-3) / 1e9 / peak, 4),
               "hbm_fraction_precode_phase": round(byt / (statistics.median(precode_ms) * 1e-3) / 1e9 / peak, 4),
               "gpu": name, "power_limit": power,
               "timing": f"median of {args.iters} CUDA-event timed calls after {args.warmup} warm-ups; phases from the library's events"}
        print(json.dumps(rec), flush=True)
        lines.append(rec)
        del hc, sym, tx, gain
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "dl_bench.jsonl"), "a") as f:
            for rec in lines:
                f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
