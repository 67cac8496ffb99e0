"""Throughput of the multi-user receiver (lsmrc_demod_frames_device_mu) against single-user MRC
(lsmrc_demod_frames_device) on the same device-resident input, alternating the two in one process.

Inputs are built on the GPU (synth.make_frames_mu_torch) and are larger than twice the 126 MB L2, so every timed call
streams its frames from HBM; the batches hold enough (frame, symbol) pairs to give every SM work (c2: 64 frames, c4: 32),
since a smaller batch measures an idle GPU for either receiver.  Per call: CUDA events around the call, >= 5 warm-ups, >= 20 timed calls, median.
One JSON line per (shape, users, detector) with the card name and power limit read in the same run.

With --soft the pair is lsmrc_demod_frames_device_mu_soft (LLRs and SINR) against lsmrc_demod_frames_device_mu on the
same input: the cost of the soft output (DESIGN.md 8f).

With --pilots comb the call runs on comb-pilot frames (one pilot symbol; DESIGN.md 8h), on c2 and on c4 at its own
S = 14 with 4, 8 and 16 users.  Where time-orthogonal pilots fit the shape (U < S) the time-pilot call on time-pilot
frames of the same shape alternates with it; decoded user-symbols/s count the data symbols of each format.

  python tools/mu_bench.py [--quick] [--soft | --pilots comb] [--out DIR]
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

HBM_PEAK_GBS = 6555.2  # measured HBM read+write peak of the B200 (DESIGN.md)
L2_BYTES = 126 << 20

# (name, A, N, C, S, U, detector, frames).  c4 with 16 users needs more than 16 symbols (16 of them are pilots): S = 20.
CASES = [
    ("c2", 64, 1024, 64, 101, 1, "zf", 64),
    ("c2", 64, 1024, 64, 101, 4, "zf", 64),
    ("c2", 64, 1024, 64, 101, 4, "mmse", 64),
    ("c2", 64, 1024, 64, 101, 8, "zf", 64),
    ("c4", 256, 4096, 288, 14, 4, "zf", 32),
    ("c4", 256, 4096, 288, 14, 4, "mmse", 32),
    ("c4", 256, 4096, 288, 14, 8, "zf", 32),
    ("c4_S20", 256, 4096, 288, 20, 16, "zf", 32),
]
SOFT_CASES = [c for c in CASES if c[5] in (4, 8) and c[0] in ("c2", "c4")]
COMB_CASES = [(tag, A, N, C, S, U, "zf", F) for (tag, A, N, C, S, F) in (("c2", 64, 1024, 64, 101, 64), ("c4", 256, 4096, 288, 14, 32))
              for U in (4, 8, 16)]


def algorithmic_bytes(A, N, S, U, qam_bits, n_pilot_sym=None):
    """per frame, P = n_pilot_sym pilot symbols (U time-orthogonal, the default, or 1 comb): samples in (8*A*S*N, CP
    not counted) + per-user channel out (8*U*A*K) + detected symbols out (8*(S-P)*U*K) + packed bits out"""
    K = N - 1
    P = U if n_pilot_sym is None else n_pilot_sym
    bits = (S - P) * U * ((K * qam_bits + 7) // 8)
    return 8 * A * S * N + 8 * U * A * K + 8 * (S - P) * U * K + bits


def soft_extra_bytes(N, S, U, qam_bits):
    """per frame, on top of algorithmic_bytes: the LLR store (4*b per user-symbol) and the SINR store (4*U*K)"""
    K = N - 1
    return 4 * qam_bits * (S - U) * U * K + 4 * U * K


def card():
    import torch

    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit", "--format=csv,noheader"], capture_output=True,
                            text=True, timeout=30).stdout.strip()
    except Exception as e:  # (reported, not guessed)
        pl = f"unknown ({e.__class__.__name__})"
    return name, pl


def time_calls(fn_a, fn_b, warmup, iters):
    import torch

    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(2)] for _ in range(2)]
    for _ in range(warmup):
        fn_a()
        fn_b()
    torch.cuda.synchronize()
    ta, tb = [], []
    for _ in range(iters):
        for fn, e, out in ((fn_a, ev[0], ta), (fn_b, ev[1], tb)):
            e[0].record()
            fn()
            e[1].record()
            e[1].synchronize()
            out.append(e[0].elapsed_time(e[1]))
    return statistics.median(ta), statistics.median(tb)


def comb_case(ofdm_b200, dev, tag, A, N, C, S, U, det, F, b, args, name, power):
    """one comb-pilot shape: comb call on comb frames, alternating with the time-pilot call on time frames when U < S"""
    import torch

    K = N - 1
    frame_bytes = 8 * S * A * (N + C)
    assert args.quick or F * frame_bytes > 2 * L2_BYTES
    layouts = ("comb", "time") if U < S else ("comb",)
    fns, outs = {}, []
    st = torch.cuda.Stream(dev)
    r = ofdm_b200.LsMrcReceiver(A, N, C, S, b)
    try:
        for lay in layouts:
            P = 1 if lay == "comb" else U
            rx, pilot, _ = ofdm_b200.synth.make_frames_mu_torch(F, A, N, C, S, b, U, dev, seed=1, snr_db=30.0, chunk=1, pilots=lay)
            comb = torch.empty((F, S - P, U, K), dtype=torch.complex64, device=dev)
            bits = torch.empty((F, S - P, U, (K * b + 7) // 8), dtype=torch.uint8, device=dev)
            hc = torch.empty((F, U, A, K), dtype=torch.complex64, device=dev)
            outs.append((rx, comb, bits, hc))

            def call(lay=lay, rx=rx, comb=comb, bits=bits, hc=hc):
                r.set_mu_pilots(lay)
                r.demod_frames_device_mu(rx, F, U, comb, bits, hc, detector=det)

            fns[lay] = call
        r.set_pilot(pilot)  # (every frame uses the same pilot: make_pilot(K, seed))
        torch.cuda.synchronize()
        with torch.cuda.stream(st):
            r.set_stream(st.cuda_stream)
            if "time" in fns:
                t_comb, t_time = time_calls(fns["comb"], fns["time"], args.warmup, args.iters)
            else:
                t_comb, t_time = time_calls(fns["comb"], lambda: None, args.warmup, args.iters)
                t_time = None
            r.set_stream(None)
    finally:
        r.close()
    rec = {"case": tag, "A": A, "N": N, "C": C, "S": S, "U": U, "detector": det, "qam_bits": b, "frames": F,
           "input_MB": round(F * frame_bytes / 1e6, 1)}
    for lay, t in (("comb", t_comb), ("time", t_time)):
        P = 1 if lay == "comb" else U
        if t is None:
            rec.update({f"ms_{lay}": None, f"data_symbols_{lay}": None, f"user_symbols_per_s_{lay}": None, f"hbm_fraction_{lay}": None})
            continue
        byt = F * algorithmic_bytes(A, N, S, U, b, P)
        rec.update({f"ms_{lay}": round(t, 4), f"data_symbols_{lay}": S - P,
                    f"user_symbols_per_s_{lay}": F * (S - P) * U * K / (t * 1e-3),
                    f"hbm_fraction_{lay}": round(byt / (t * 1e-3) / 1e9 / HBM_PEAK_GBS, 4)})
    rec.update({"gpu": name, "power_limit": power,
                "timing": f"median of {args.iters} CUDA-event timed calls after {args.warmup} warm-ups"
                          + (", comb and time alternating" if t_time is not None else " (time pilots need U < S)")})
    del outs
    torch.cuda.empty_cache()
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--quick", action="store_true", help="first two cases only, one frame each (rehearsal)")
    ap.add_argument("--soft", action="store_true", help="soft multi-user call against the hard one instead of MU against MRC")
    ap.add_argument("--pilots", choices=("time", "comb"), default="time",
                    help="comb: comb-pilot frames, alternating with time pilots where they fit, instead of MU against MRC")
    ap.add_argument("--out", default=None, help="also append the JSON lines to DIR/mu_bench.jsonl")
    args = ap.parse_args()
    if args.soft and args.pilots == "comb":
        raise SystemExit("--soft and --pilots comb are separate runs")
    import torch

    import ofdm_b200

    if not torch.cuda.is_available():
        raise SystemExit("mu_bench needs a CUDA GPU")
    dev = torch.device("cuda:0")
    name, power = card()
    b = 4
    lines = []
    cases = SOFT_CASES if args.soft else COMB_CASES if args.pilots == "comb" else CASES
    for (tag, A, N, C, S, U, det, F) in (cases[:2] if args.quick else cases):
        if args.pilots == "comb":
            rec = comb_case(ofdm_b200, dev, tag, A, N, C, S, U, det, 1 if args.quick else F, b, args, name, power)
            print(json.dumps(rec), flush=True)
            lines.append(rec)
            continue
        K = N - 1
        frame_bytes = 8 * S * A * (N + C)
        if args.quick:
            F = 1
        else:
            assert F * frame_bytes > 2 * L2_BYTES
        rx, pilot, _ = ofdm_b200.synth.make_frames_mu_torch(F, A, N, C, S, b, U, dev, seed=1, snr_db=30.0, chunk=1)
        comb_mu = torch.empty((F, S - U, U, K), dtype=torch.complex64, device=dev)
        bits_mu = torch.empty((F, S - U, U, (K * b + 7) // 8), dtype=torch.uint8, device=dev)
        hc_mu = torch.empty((F, U, A, K), dtype=torch.complex64, device=dev)
        comb_su = torch.empty((F, S - 1, K), dtype=torch.complex64, device=dev)
        bits_su = torch.empty((F, S - 1, (K * b + 7) // 8), dtype=torch.uint8, device=dev)
        hc_su = torch.empty((F, A, K), dtype=torch.complex64, device=dev)
        nv = 0.001 if det == "mmse" or args.soft else 0.0
        if args.soft:
            llr = torch.empty((F, S - U, U, K, b), dtype=torch.float32, device=dev)
            sinr = torch.empty((F, U, K), dtype=torch.float32, device=dev)
        torch.cuda.synchronize()
        st = torch.cuda.Stream(dev)  # (a stream of its own: handle 0 would select the receiver's internal stream)
        with ofdm_b200.LsMrcReceiver(A, N, C, S, b) as r, torch.cuda.stream(st):
            r.set_pilot(pilot)
            r.set_stream(st.cuda_stream)

            def mu():
                r.demod_frames_device_mu(rx, F, U, comb_mu, bits_mu, hc_mu, detector=det, noise_var=nv)

            def su():
                r.demod_frames_device(rx, F, comb_su, bits_su, hc_su)

            def soft():
                r.demod_frames_device_mu_soft(rx, F, U, comb_mu, llr, bits_mu, hc_mu, sinr, detector=det, noise_var=nv)

            if args.soft:
                t_soft, t_mu = time_calls(soft, mu, args.warmup, args.iters)
            else:
                t_mu, t_su = time_calls(mu, su, args.warmup, args.iters)
            r.set_stream(None)
        byt = F * algorithmic_bytes(A, N, S, U, b)
        if args.soft:
            sbyt = byt + F * soft_extra_bytes(N, S, U, b)
            rec = {"case": tag, "A": A, "N": N, "C": C, "S": S, "U": U, "detector": det, "qam_bits": b, "frames": F,
                   "ms_soft": round(t_soft, 4), "ms_hard": round(t_mu, 4), "soft_over_hard": round(t_soft / t_mu, 4),
                   "llr_bytes_over_input": round(soft_extra_bytes(N, S, U, b) / (8 * A * S * N), 4),
                   "alg_GBps_soft": round(sbyt / (t_soft * 1e-3) / 1e9, 1),
                   "hbm_fraction_soft": round(sbyt / (t_soft * 1e-3) / 1e9 / HBM_PEAK_GBS, 4), "gpu": name, "power_limit": power,
                   "timing": f"median of {args.iters} CUDA-event timed calls after {args.warmup} warm-ups, soft and hard alternating"}
            print(json.dumps(rec), flush=True)
            lines.append(rec)
            del rx, comb_mu, bits_mu, hc_mu, comb_su, bits_su, hc_su, llr, sinr
            torch.cuda.empty_cache()
            continue
        rec = {"case": tag, "A": A, "N": N, "C": C, "S": S, "U": U, "detector": det, "qam_bits": b, "frames": F,
               "input_MB": round(F * frame_bytes / 1e6, 1), "ms_mu": round(t_mu, 4), "ms_mrc": round(t_su, 4),
               "antenna_samples_per_s": F * S * A * (N + C) / (t_mu * 1e-3),
               "alg_GBps": round(byt / (t_mu * 1e-3) / 1e9, 1),
               "hbm_fraction": round(byt / (t_mu * 1e-3) / 1e9 / HBM_PEAK_GBS, 4),
               "ratio_to_mrc": round(t_su / t_mu, 4), "gpu": name, "power_limit": power,
               "timing": f"median of {args.iters} CUDA-event timed calls after {args.warmup} warm-ups, alternating with MRC"}
        print(json.dumps(rec), flush=True)
        lines.append(rec)
        del rx, comb_mu, bits_mu, hc_mu, comb_su, bits_su, hc_su
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "mu_bench.jsonl"), "a") as f:
            for rec in lines:
                f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
