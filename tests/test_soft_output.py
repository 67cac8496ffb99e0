"""Single-user soft output against float64 references, on every launch path of the data kernels.

lsmrc_demod_frames_device_soft gets its LLRs from the epilogue every single-user data kernel shares (mrc_finish); which
kernel runs it depends on the batch and the launch policy (launch_frames / launch_impl in csrc/lsmrc_capi.cu).  The
hard bits come out right even when the soft values are wrong, so every route is checked here element by element:

  * ref_chain64 restates the receive chain in plain numpy float64 (CP strip, FFT, LS estimate, MRC, max-log LLRs),
    independently of oracle/;
  * llr_bound_ratio is a per-element comparator: the error an fp32 implementation may make on bit j of (f, s, k) scales
    with the RMS of the antenna rows that went into it, not with the largest LLR of the array;
  * llr64 / noise_var64 apply the header's formulas (include/ofdm_lsmrc.h) to given arrays, for the stand-alone
    lsmrc_llr_from_combined and lsmrc_estimate_noise_var.

The CPU tests pin the references and show that the comparator accepts a real fp32 implementation (the C oracle) and
rejects small, plausible kernel mistakes.  The GPU tests run each kernel route with LLRs on."""
import json
import os
import tempfile
import types

import numpy as np
import pytest

from util import assert_bits_match

TAU = 1e-5                                                      # the project's fp32 parity tolerance
A_EXACT = {2: 1 / np.sqrt(2.0), 4: 1 / np.sqrt(10.0), 6: 1 / np.sqrt(42.0)}
U32 = 2.0 ** -24                                                # unit roundoff of float32
SNR = {2: 10.0, 4: 15.0, 6: 20.0}


def _bin_to_asc(v):
    K = v.shape[-1]
    return np.roll(v, (K + 1) // 2, axis=-1)                    # = synth.bin_to_asc


def amp_consts(b):
    """per bit j: the sum of the constants in that bit's max-log formula (0 for the two sign bits)"""
    a = A_EXACT[b]
    return np.array({2: [0, 0], 4: [0, 0, 2 * a, 2 * a], 6: [0, 0, 4 * a, 4 * a, 6 * a, 6 * a]}[b], np.float64)


def soft64(y, rho, b):
    """max-log piecewise-linear LLRs (soft_symbol in csrc/lsmrc_kernels.cuh) in float64 with the exact constants:
    y complex [..., K] ascending frequency, rho = sum|H|^2 / noise_var broadcastable to y -> [..., K, b]"""
    a = A_EXACT[b]
    g = 4 * a * np.asarray(rho, np.float64)
    re, im = np.asarray(y).real.astype(np.float64), np.asarray(y).imag.astype(np.float64)
    out = [g * re, g * im]
    if b == 4:
        out += [g * (2 * a - np.abs(re)), g * (2 * a - np.abs(im))]
    elif b == 6:
        out += [g * (4 * a - np.abs(re)), g * (4 * a - np.abs(im)),
                g * (2 * a - np.abs(np.abs(re) - 4 * a)), g * (2 * a - np.abs(np.abs(im) - 4 * a))]
    return np.stack(out, axis=-1)


def llr64(y, E_bin, nv_per_frame, b):
    """lsmrc_llr_from_combined in float64: y [F,D,K] ascending frequency, E_bin [F,K] = sum|H|^2 in FFT-bin order,
    nv_per_frame [F] -> [F,D,K,b]"""
    nv = np.asarray(nv_per_frame, np.float64).reshape(-1)
    rho = _bin_to_asc(np.asarray(E_bin, np.float64)) / nv[:, None]
    return soft64(np.asarray(y, np.complex128), rho[:, None, :], b)


def _slice64(u, b):
    """nearest constellation level of one axis, exact levels and decision thresholds"""
    a = A_EXACT[b]
    top = {2: 1, 4: 3, 6: 7}[b]
    k = np.clip(2 * np.floor(np.abs(u) / (2 * a)) + 1, 1, top)
    return np.where(u < 0, -k * a, k * a)


def noise_var64(y, E_bin, b):
    """lsmrc_estimate_noise_var in float64: mean over (s, i) of sum|H|^2[bin(i)] * |y - slice(y)|^2, per frame [F]"""
    y = np.asarray(y, np.complex128)
    r2 = (y.real - _slice64(y.real, b)) ** 2 + (y.imag - _slice64(y.imag, b)) ** 2
    e = _bin_to_asc(np.asarray(E_bin, np.float64))
    return (r2 * e[:, None, :]).sum(axis=(1, 2)) / (y.shape[1] * y.shape[2])


def ref_chain64(rx, pilot_asc, cp, b, noise_var):
    """The whole single-user receive chain in complex128, frame by frame.  rx [F,S,A,N+C] -> dict
      y    [F,S-1,K] combined symbols, ascending frequency     E [F,K] sum_a |H|^2, FFT-bin order
      llr  [F,S-1,K,b] max-log LLRs with rho = E / noise_var   nv  the noise variance used
      u    [F,S-1,K] sum_a (|H_ak| + r_H,a) (|Y_sak| + r_Y,sa)  w [F,K] sum_a (|H_ak| + r_H,a)^2   (ascending frequency)
    where r is the RMS of that antenna row over the K bins (the scale of an fp32 FFT's error in the row)."""
    rx = np.asarray(rx)
    F, S, A, NC = rx.shape
    K = NC - cp - 1
    x_bin = np.roll(np.asarray(pilot_asc).astype(np.complex128), -((K + 1) // 2))       # = synth.asc_to_bin
    y = np.empty((F, S - 1, K), np.complex128)
    E = np.empty((F, K))
    u = np.empty((F, S - 1, K))
    w = np.empty((F, K))
    for f in range(F):
        Z = np.fft.fft(rx[f, :, :, cp:].astype(np.complex128), axis=-1)[..., 1:]          # [S,A,K], bins 1..N-1
        H = Z[0] / x_bin
        Y = Z[1:]
        E[f] = (np.abs(H) ** 2).sum(0)
        y[f] = (Y * np.conj(H)).sum(1) / E[f]
        hh = np.abs(H) + np.sqrt((np.abs(H) ** 2).mean(-1))[:, None]                     # [A,K]
        yy = np.abs(Y) + np.sqrt((np.abs(Y) ** 2).mean(-1))[..., None]                   # [S-1,A,K]
        u[f] = np.einsum("ak,sak->sk", hh, yy)
        w[f] = (hh ** 2).sum(0)
    y, u, w = _bin_to_asc(y), _bin_to_asc(u), _bin_to_asc(w)
    nv = float(noise_var)
    return {"y": y, "E": E, "llr": soft64(y, (_bin_to_asc(E) / nv)[:, None, :], b), "nv": nv, "u": u, "w": w}


def llr_bound_ratio(got, ref, b, tau=TAU):
    """|got - llr64| over the per-element bound
        tau * (4a / sigma^2) * ( u[f,s,k] + c_j * w[f,k] ),   c_j = amp_consts(b)[j]
    (float64, same shape as got; non-finite values give inf)"""
    got = np.asarray(got, np.float64)
    assert got.shape == ref["llr"].shape, (got.shape, ref["llr"].shape)
    bound = tau * (4 * A_EXACT[b] / ref["nv"]) * (ref["u"][..., None] + amp_consts(b) * ref["w"][:, None, :, None])
    r = np.abs(got - ref["llr"]) / bound
    r[~np.isfinite(got)] = np.inf
    return r


def assert_llrs_within_bound(got, ref, b, what):
    """every element inside its bound; the failure names the worst (f, s, k, j).  Returns the largest ratio."""
    r = llr_bound_ratio(got, ref, b)
    worst = np.unravel_index(int(np.argmax(r)), r.shape)
    m = float(r[worst])
    assert m <= 1.0, (f"{what}: LLR outside its fp32 error bound at (f, s, k, j) = {tuple(int(i) for i in worst)}: ratio {m:.3g}, "
                      f"got {float(np.asarray(got)[worst])!r}, float64 {float(ref['llr'][worst])!r}; "
                      f"{int((r > 1).sum())} of {r.size} elements out of bound")
    return m


def ref_bits64(ref, b):
    """hard decisions of the float64 chain, packed like d_bits (bit 1 <=> LLR < 0: the max-log form's sign is exactly
    the demapper's decision)"""
    F, D, K = ref["y"].shape
    hard = (ref["llr"] < 0).astype(np.uint8).reshape(F, D, K * b)
    return np.packbits(hard, axis=-1, bitorder="little")


def ulp_scale(y, E_bin, nv_per_frame, b):
    """per element the magnitude the fp32 evaluation of the LLR formula rounds against:
    4a * rho * (|component| + c_j) -- the operands of its one subtraction chain and its products"""
    nv = np.asarray(nv_per_frame, np.float64).reshape(-1)
    rho = (_bin_to_asc(np.asarray(E_bin, np.float64)) / nv[:, None])[:, None, :]
    y = np.asarray(y, np.complex128)
    comp = np.stack([np.abs(y.real), np.abs(y.imag)] * (b // 2), axis=-1)
    return (4 * A_EXACT[b] * rho)[..., None] * (comp + amp_consts(b))


FORMULA_ULPS = 8   # float32 rounding steps allowed between the fp32 formula and llr64 (see test_llr64_pins_the_fp32_formula)


def formula_ulps(got, y, E_bin, nv_per_frame, b):
    """|got - llr64| in float32 rounding steps of ulp_scale (a zero component's sign bits must be exactly 0)"""
    d = np.abs(np.asarray(got, np.float64) - llr64(y, E_bin, nv_per_frame, b))
    s = U32 * ulp_scale(y, E_bin, nv_per_frame, b)
    return np.divide(d, s, out=np.where(d > 0, np.inf, 0.0), where=s > 0)


def soft_inputs(F, D, N, b, seed):
    """synthetic combined symbols [F,D,K] complex64 (ascending frequency), sum|H|^2 [F,K] float32 log-uniform over
    1e-3..1e3 per bin, and a different noise variance per frame: constellation points plus noise whose level differs
    per frame, with about 5 % of the components replaced by zero, the kernel's fp32 constellation levels (k * a as
    float32) and its decision thresholds"""
    import ofdm_b200

    rng = np.random.default_rng(seed)
    K = N - 1
    qam_map_indices = ofdm_b200.synth.qam_map_indices
    sigma = 0.02 + 0.03 * (np.arange(F) % 7) + 1e-3 * np.arange(F)
    idx = rng.integers(0, 1 << b, size=(F, D, K))
    y = qam_map_indices(idx, b) + sigma[:, None, None] * (rng.standard_normal((F, D, K)) + 1j * rng.standard_normal((F, D, K))) / np.sqrt(2)
    y = y.astype(np.complex64)
    af = np.float32(A_EXACT[b])
    edges = [np.float32(0.0)] + [np.float32(k) * af for k in range(1, {2: 2, 4: 4, 6: 8}[b])]   # levels (odd k), LLR thresholds (even k)
    if b == 4:
        edges.append(np.float32(0.6324555320336759))                                           # hard-demap thresholds
    if b == 6:
        t4, t2 = np.float32(0.6172133998483676), np.float32(0.3086066999241838)
        edges += [t4, t2, np.float32(t4 + t2), np.float32(t4 - t2)]
    edges = np.array(edges, np.float32)
    parts = y.view(np.float32).reshape(F, D, K, 2)
    hit = rng.random(parts.shape) < 0.05
    pick = edges[rng.integers(0, len(edges), parts.shape)] * np.where(rng.random(parts.shape) < 0.5, np.float32(-1), np.float32(1))
    parts[hit] = pick[hit]
    E = (10.0 ** rng.uniform(-3.0, 3.0, size=(F, K))).astype(np.float32)
    nv = (10.0 ** rng.uniform(-2.0, 0.0, size=F)).astype(np.float32)
    return y, E, nv


# ------------------------------------------------------------------------------------------------ CPU
def _fp32_result(ofdm, oracle, A, N, C, S, b, F, seed):
    d = ofdm.synth.make_frames(F, A, N, C, S, b, snr_db=SNR[b], seed=seed)
    nv = float(np.float32((N - 1) / N * 10.0 ** (-SNR[b] / 10.0)))
    ref32 = oracle.demod_frames(d["rx"], d["pilot_asc"], b, C)
    llr32 = oracle.soft_demap(ref32["combined"], ref32["hsqrd"], b, nv)
    return d, ref32, llr32, ref_chain64(d["rx"], d["pilot_asc"], C, b, nv)


@pytest.mark.parametrize("b", [2, 4, 6])
@pytest.mark.parametrize("dims", [(8, 64, 16, 6, 3), (16, 1024, 64, 4, 2), (8, 4096, 288, 3, 2)], ids=["N64", "N1024", "N4096"])
def test_comparator_accepts_the_fp32_oracle(ofdm, oracle, dims, b):
    """the fp32 C oracle's combined symbols + oracle.soft_demap are a real fp32 implementation of the chain: the
    per-element bound must hold with room to spare"""
    A, N, C, S, F = dims
    _, ref32, llr32, ref = _fp32_result(ofdm, oracle, A, N, C, S, b, F, seed=N + b)
    m = assert_llrs_within_bound(llr32, ref, b, "fp32 oracle")
    print(f"fp32 oracle, N={N} b={b}: largest ratio to the bound {m:.3g}")
    assert m < 0.25
    assert np.abs(ref32["combined"] - ref["y"]).max() <= 1e-5 * np.abs(ref["y"]).max()   # (the chains agree)


def _mutations(b):
    names = ["rho_neighbour_bin", "frequency_roll", "row_of_next_symbol", "row_of_next_frame", "scale_one_element",
             "flip_one_sign"]
    return names + (["swap_amplitude_bits"] if b >= 4 else [])


@pytest.mark.parametrize("b,mutation", [(b, m) for b in (2, 4, 6) for m in _mutations(b)])
def test_comparator_rejects_plausible_kernel_mistakes(ofdm, oracle, b, mutation):
    A, N, C, S, F = 8, 256, 32, 5, 3
    _, ref32, llr32, ref = _fp32_result(ofdm, oracle, A, N, C, S, b, F, seed=7 + b)
    assert llr_bound_ratio(llr32, ref, b).max() <= 1.0
    bad = llr32.copy()
    where = None
    if mutation == "rho_neighbour_bin":
        bad = oracle.soft_demap(ref32["combined"], np.roll(ref32["hsqrd"], 1, axis=-1), b, ref["nv"])
    elif mutation == "frequency_roll":
        bad = np.roll(llr32, 1, axis=2)
    elif mutation == "row_of_next_symbol":
        bad[1, 2] = llr32[1, 3]
    elif mutation == "row_of_next_frame":
        bad[1, 2] = llr32[2, 2]
    elif mutation == "swap_amplitude_bits":
        k = 100
        bad[0, 1, k, [2, 3]] = llr32[0, 1, k, [3, 2]]
        where = None if llr32[0, 1, k, 2] == llr32[0, 1, k, 3] else (0, 1, k)
    else:
        where = np.unravel_index(int(np.argmax(np.abs(llr32))), llr32.shape)
        bad[where] = llr32[where] * np.float32(1 + 1e-3) if mutation == "scale_one_element" else -llr32[where]
    r = llr_bound_ratio(bad, ref, b)
    if where is not None:
        worst = np.unravel_index(int(np.argmax(r)), r.shape)
        assert worst[:len(where)] == tuple(where), (worst, where)
    with pytest.raises(AssertionError, match=r"outside its fp32 error bound at \(f, s, k, j\)"):
        assert_llrs_within_bound(bad, ref, b, mutation)


@pytest.mark.parametrize("b", [2, 4, 6])
def test_llr64_pins_the_fp32_formula(oracle, b):
    """llr64 (exact constants, float64) and oracle.soft_demap (the fp32 formula the kernels share, same constants and
    operation order) agree to a few float32 rounding steps of the formula's operands, element by element -- including
    components on the decision thresholds and on the fp32 constellation levels, where the amplitude bits cancel"""
    F, D, N = 5, 3, 1024
    y, E, nv = soft_inputs(F, D, N, b, seed=40 + b)
    got = np.stack([oracle.soft_demap(y[f:f + 1], E[f:f + 1], b, float(nv[f]))[0] for f in range(F)])
    ulps = formula_ulps(got, y, E, nv, b)
    print(f"b={b}: largest difference {ulps.max():.2f} float32 rounding steps")
    assert ulps.max() <= FORMULA_ULPS, ulps.max()
    # tight enough to see rho off by 16 float32 steps
    assert formula_ulps(got * np.float32(1 + 2 ** -20), y, E, nv, b).max() > FORMULA_ULPS


def test_noise_var64_is_the_header_formula(ofdm, oracle):
    """noise_var64 against the C oracle's float64 accumulation of the same definition; exact constellation points give 0"""
    for b in (2, 4, 6):
        y, E, _ = soft_inputs(4, 6, 256, b, seed=60 + b)
        assert np.allclose(noise_var64(y, E, b), oracle.noise_var(y, E, b), rtol=1e-6, atol=0)
        pts = ofdm.synth.qam_map_indices(np.arange(1 << b), b)
        assert noise_var64(np.tile(pts, (1, 2, 1)), np.ones((1, pts.size)), b)[0] < 1e-30


# ------------------------------------------------------------------------------------------------ GPU
GUARD = 4096          # sentinel elements after every output buffer


def _guarded(n, dtype, fill, dev):
    """(whole buffer, its first n elements): the rest is a guard tail that must stay as filled"""
    import torch

    buf = torch.full((n + GUARD,), fill, dtype=dtype, device=dev)
    return buf, buf[:n]


def _tail_intact(buf, n, fill_bits, view):
    return bool((buf[n:].cpu().numpy().view(view) == fill_bits).all())


def _frames(ofdm, dims, seed, dev):
    """realistic frames built on the device: rx [F,S,A,N+C] complex64 tensor and the pilot"""
    A, N, C, S, b, F = dims
    cfg = types.SimpleNamespace(n_ant=A, fft_size=N, cp_len=C, n_sym=S, qam_bits=b, seed=seed, snr_db=SNR[b])
    rx, pilot, _ = ofdm.synth.make_frames_torch(F, cfg, dev, seed=seed, snr_db=SNR[b], chunk=16)
    return rx, pilot


def _noise_var_of(N, b):
    """noise variance per antenna and subcarrier after the FFT of make_frames_torch's AWGN"""
    return float(np.float32((N - 1) / N * 10.0 ** (-SNR[b] / 10.0)))


# (id, (A, N, C, S, b, F), launch policy for small batches (set_oneshot), single launch on (set_one_launch_frames), kernel
# family, antenna split).  The routes follow from launch_frames / launch_impl in csrc/lsmrc_capi.cu; the route-map test
# below checks each of them with torch.profiler.
ROUTES = [
    # one-launch kernel (MODE_ONESHOT): latency plans at 64..256 points, the throughput plans from 512 up
    ("oneshot_64", (4, 64, 16, 6, 2, 3), 2, True, "oneshot", None),
    ("oneshot_128", (8, 128, 16, 5, 4, 2), 2, True, "oneshot", None),
    ("oneshot_256", (8, 256, 32, 4, 6, 1), 2, True, "oneshot", None),
    ("oneshot_512", (12, 512, 128, 4, 6, 1), 2, True, "oneshot", None),
    ("oneshot_1024", (6, 1024, 64, 5, 4, 1), 2, True, "oneshot", None),
    ("oneshot_2048", (3, 2048, 144, 3, 2, 1), 2, True, "oneshot", None),
    ("oneshot_4096", (2, 4096, 288, 3, 6, 1), 2, True, "oneshot", None),
    # generic data kernel (MODE_DATA) on the plans up to 512 points, antennas split over teams or not
    ("data_64_split", (4, 64, 16, 16, 2, 3), 0, True, "data", True),
    ("data_64", (4, 64, 16, 16, 2, 300), 0, True, "data", False),
    ("data_128_split", (16, 128, 32, 9, 4, 1), 0, True, "data", True),
    ("data_512", (4, 512, 32, 7, 2, 600), 0, True, "data", False),
    # 1024 points: the H-ring data kernel with bulk-copied sample rows (even prefix) and without (odd prefix)
    ("ring_1024_bulk", (16, 1024, 64, 6, 4, 7), 0, True, "data_xt", None),
    ("ring_1024_plain", (6, 1024, 9, 3, 6, 2), 0, True, "data", None),
    # 2048 points, one (frame, symbol) pair per team is too few: the generic kernel with the antennas split
    ("data_2048_split", (4, 2048, 144, 3, 4, 1), 0, True, "data", True),
    # shuffle-stage plans, large batches, single launch off: the dedicated data kernel, even and odd prefix
    ("data_sh_2048", (3, 2048, 144, 10, 4, 70), 0, False, "data_sh", None),
    ("data_sh_2048_odd", (5, 2048, 7, 4, 6, 161), 0, False, "data_sh", None),
    ("data_sh_4096", (3, 4096, 288, 6, 6, 60), 0, False, "data_sh", None),
    ("data_sh_4096_odd", (2, 4096, 33, 3, 2, 130), 0, False, "data_sh", None),
    # ... single launch on: pilot and data items in one persistent kernel (the E_CG epilogue); the third case has
    # two antenna groups per frame, the second an odd prefix
    ("frames_sh_2048", (3, 2048, 144, 8, 4, 140), 2, True, "frames_sh", None),
    ("frames_sh_4096_odd", (2, 4096, 33, 3, 2, 230), 2, True, "frames_sh", None),
    ("frames_sh_4096_groups", (32, 4096, 288, 4, 6, 150), 2, True, "frames_sh", None),
]
ROUTE_IDS = [r[0] for r in ROUTES]


def _receiver(ofdm, dims, pilot, policy, one_launch):
    A, N, C, S, b, F = dims
    r = ofdm.LsMrcReceiver(A, N, C, S, b)
    r.set_pilot(pilot)
    r.set_oneshot(policy)
    r.set_one_launch_frames(one_launch)
    return r


def _kernel_launches(fn):
    """(demangled name, grid) of every CUDA kernel fn() launches, from torch.profiler (CUDA activity only, in-process;
    the trace goes to a temporary directory)"""
    import torch
    from torch.profiler import ProfilerActivity, profile

    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as fh:
            events = json.load(fh)["traceEvents"]
    return [(e["name"], tuple(e.get("args", {}).get("grid", ()))) for e in events if e.get("cat") == "kernel"]


def _family(name):
    """(family, N, TEAMS) of a single-user data-path kernel name, None for anything else.  Families: oneshot
    (lsmrc_kernel MODE_ONESHOT), data / data_xt (lsmrc_kernel MODE_DATA without / with bulk copies), data_sh, frames_sh"""
    import re

    m = re.search(r"(lsmrc_kernel|lsmrc_data_sh|lsmrc_frames_sh)<lsmrc::Plan<(\d+), \d+, \d+, \d+, (\d+)[^>]*>, (\d+)"
                  r"(?:, \d+, (true|false))?>", name)
    if not m:
        return None
    kern, n, teams, mode, xt = m.group(1), int(m.group(2)), int(m.group(3)), int(m.group(4)), m.group(5)
    if kern == "lsmrc_data_sh":
        return ("data_sh", n, teams)
    if kern == "lsmrc_frames_sh":
        return ("frames_sh", n, teams)
    fam = {3: "oneshot", 1: "data_xt" if xt == "true" else "data"}.get(mode)
    return (fam, n, teams) if fam else None


@pytest.mark.gpu
def test_gpu_route_map(ofdm):
    """every case of ROUTES runs its soft call through the kernel it is listed for (and, where it says so, with the
    antennas split over teams: more CTAs than one team per (frame, symbol) pair would need); together they reach every
    single-user data kernel family with LLRs on"""
    import torch

    dev = torch.device("cuda:0")
    seen = set()
    table = []
    for rid, dims, policy, one_launch, fam, split in ROUTES:
        A, N, C, S, b, F = dims
        K = N - 1
        rx, pilot = _frames(ofdm, dims, seed=3, dev=dev)
        comb = torch.empty((F, S - 1, K, 2), device=dev)
        llr = torch.empty((F, S - 1, K, b), device=dev)
        torch.cuda.synchronize()
        with _receiver(ofdm, dims, pilot, policy, one_launch) as r:
            def call():
                r.demod_frames_device_soft(rx, F, comb, llr, _noise_var_of(N, b))
                r.sync()

            call()                                       # (first call: channel state allocated)
            launches = _kernel_launches(call)
        fams = [(_family(n), g) for n, g in launches if _family(n)]
        table.append(f"{rid}: " + ", ".join(f"{f[0]}/{f[1]} grid {g}" for f, g in fams))
        hits = [(f, g) for f, g in fams if f[0] == fam and f[1] == N]
        assert hits, f"{rid}: expected {fam} at {N} points, launched {[n for n, _ in launches]}"
        if split is not None:
            (_, _, teams), grid = hits[0]
            assert grid, f"{rid}: the trace has no grid for {hits[0]}"
            pairs_per_cta = -(-(F * (S - 1)) // teams)
            assert (grid[0] > pairs_per_cta) == split, (rid, grid, pairs_per_cta)
        seen.add((fam, N))
        if fam == "data" and N <= 512:
            seen.add(("data", "<=512", "split" if split else "no split"))
    print("\n".join(table))
    want = {("oneshot", n) for n in (64, 128, 256, 512, 1024, 2048, 4096)} | \
        {("data", "<=512", "split"), ("data", "<=512", "no split"), ("data_xt", 1024), ("data", 1024), ("data", 2048),
         ("data_sh", 2048), ("data_sh", 4096), ("frames_sh", 2048), ("frames_sh", 4096)}
    assert want <= seen, want - seen


@pytest.mark.gpu
@pytest.mark.parametrize("route", ROUTES, ids=ROUTE_IDS)
def test_gpu_soft_output_on_every_route(ofdm, route):
    """On each route, with NaN-filled outputs followed by a guard tail:
      1. every in-range LLR is written and finite, and no output writes past its end;
      2. d_combined and d_bits are byte-identical to the hard call's (same input, same launch policy);
      3. the epilogue's LLRs are bit-identical to lsmrc_llr_from_combined on the soft call's combined symbols, the hard
         call's sum|H|^2 and the same noise variance (both: one correctly rounded reciprocal, one product, soft_symbol);
      4. every LLR is inside its per-element fp32 bound around the float64 chain;
      5. the hard bits match the float64 chain's decisions up to threshold ties."""
    import torch

    rid, dims, policy, one_launch, fam, _ = route
    A, N, C, S, b, F = dims
    K, D = N - 1, S - 1
    nv = _noise_var_of(N, b)
    dev = torch.device("cuda:0")
    rx, pilot = _frames(ofdm, dims, seed=11, dev=dev)
    n_c, n_b, n_l = F * D * K * 2, F * D * ((K * b + 7) // 8), F * D * K * b
    comb_h_buf, comb_h = _guarded(n_c, torch.float32, float("nan"), dev)
    bits_h_buf, bits_h = _guarded(n_b, torch.uint8, 0x5A, dev)
    hsq = torch.full((F, K), float("nan"), device=dev)
    comb_s_buf, comb_s = _guarded(n_c, torch.float32, float("nan"), dev)
    bits_s_buf, bits_s = _guarded(n_b, torch.uint8, 0xA5, dev)
    llr_buf, llr = _guarded(n_l, torch.float32, float("nan"), dev)
    llr_alone_buf, llr_alone = _guarded(n_l, torch.float32, float("nan"), dev)
    nv_dev = torch.full((F,), nv, device=dev)
    torch.cuda.synchronize()                        # (the fills run on torch's stream, the receiver on its own)
    with _receiver(ofdm, dims, pilot, policy, one_launch) as r:
        r.demod_frames_device(rx, F, comb_h, bits_h, None, hsq)
        r.sync()
        n_one, n_fused = r.oneshot_count(), r.one_launch_frames_count()
        r.demod_frames_device_soft(rx, F, comb_s, llr, nv, bits_s)
        r.sync()
        assert (r.oneshot_count() - n_one, r.one_launch_frames_count() - n_fused) == \
            (int(fam == "oneshot"), int(fam == "frames_sh")), rid
        r.llr_from_combined(comb_s, hsq, nv_dev, F, llr_alone)
        r.sync()
    nan_bits = np.float32(np.nan).view(np.uint32)
    for name, buf, n, fill, view in [("llr", llr_buf, n_l, nan_bits, np.uint32), ("combined", comb_s_buf, n_c, nan_bits, np.uint32),
                                     ("bits", bits_s_buf, n_b, 0xA5, np.uint8), ("hard combined", comb_h_buf, n_c, nan_bits, np.uint32),
                                     ("hard bits", bits_h_buf, n_b, 0x5A, np.uint8)]:
        assert _tail_intact(buf, n, fill, view), f"{rid}: {name} written past its end"
    got = llr.view(F, D, K, b).cpu().numpy()
    assert np.isfinite(got).all(), f"{rid}: {int((~np.isfinite(got)).sum())} LLRs not written or not finite"
    c_s, c_h = comb_s.cpu().numpy(), comb_h.cpu().numpy()
    assert np.isfinite(c_s).all() and np.isfinite(hsq.cpu().numpy()).all()
    assert c_s.tobytes() == c_h.tobytes(), f"{rid}: LLRs on changed d_combined"
    assert bits_s.cpu().numpy().tobytes() == bits_h.cpu().numpy().tobytes(), f"{rid}: LLRs on changed d_bits"
    alone = llr_alone.view(F, D, K, b).cpu().numpy()
    same = got.view(np.uint32) == alone.view(np.uint32)
    assert same.all(), (f"{rid}: epilogue and lsmrc_llr_from_combined differ on {int((~same).sum())} LLRs, first at "
                        f"{tuple(int(i) for i in np.argwhere(~same)[0])}")
    ref = ref_chain64(rx.cpu().numpy(), pilot, C, b, nv)
    m = assert_llrs_within_bound(got, ref, b, rid)
    print(f"{rid}: largest LLR error / bound {m:.3g}")
    comb_c = c_s.reshape(F, D, K, 2).view(np.complex64)[..., 0]
    assert_bits_match(bits_s.view(F, D, -1).cpu().numpy(), ref_bits64(ref, b), ref["y"], b, rid, got_combined=comb_c)


# (F, S - 1, N, b): every F in {1, 8, 9, 37} (k_noise_frames: 8 frames per block), S - 1 in {1, 32, 33, 100} (its warp
# loop over rows), N in {64, 1024, 4096}, b in {2, 4, 6}; the last two cases have more than 148 * 32 * 256 = 1,212,416
# symbols, so k_llr_rows' grid-stride loop runs
SWEEP = [(1, 1, 64, 2), (8, 32, 1024, 4), (9, 33, 64, 6), (37, 100, 64, 4), (1, 100, 4096, 6), (9, 1, 4096, 2),
         (37, 33, 1024, 6), (4, 100, 4096, 2)]
SWEEP_IDS = ["F{}_D{}_N{}_b{}".format(*c) for c in SWEEP]


@pytest.mark.gpu
@pytest.mark.parametrize("case", SWEEP, ids=SWEEP_IDS)
def test_gpu_llr_from_combined_alone(ofdm, oracle, case):
    """lsmrc_llr_from_combined on synthetic inputs (per-bin sum|H|^2 over six decades, a noise variance per frame,
    components on thresholds and fp32 levels): within FORMULA_ULPS float32 rounding steps of llr64 per element, and bit
    for bit the fp32 formula of the C oracle (same constants, same operation order)"""
    import torch

    F, D, N, b = case
    K = N - 1
    y, E, nv = soft_inputs(F, D, N, b, seed=F * 1000 + D * 10 + b)
    dev = torch.device("cuda:0")
    d_y = torch.from_numpy(y).to(dev)
    d_e = torch.from_numpy(E).to(dev)
    d_nv = torch.from_numpy(nv).to(dev)
    n = F * D * K * b
    buf, out = _guarded(n, torch.float32, float("nan"), dev)
    torch.cuda.synchronize()
    with ofdm.LsMrcReceiver(1, N, 0, D + 1, b) as r:
        r.llr_from_combined(d_y, d_e, d_nv, F, out)
        r.sync()
    assert _tail_intact(buf, n, np.float32(np.nan).view(np.uint32), np.uint32)
    got = out.view(F, D, K, b).cpu().numpy()
    assert np.isfinite(got).all()
    ulps = formula_ulps(got, y, E, nv, b)
    worst = np.unravel_index(int(np.argmax(ulps)), ulps.shape)
    assert ulps[worst] <= FORMULA_ULPS, (tuple(int(i) for i in worst), float(ulps[worst]))
    for f in range(F):
        want = oracle.soft_demap(y[f:f + 1], E[f:f + 1], b, float(nv[f]))[0]
        assert got[f].view(np.uint32).tobytes() == want.view(np.uint32).tobytes(), f


@pytest.mark.gpu
@pytest.mark.parametrize("case", SWEEP, ids=SWEEP_IDS)
def test_gpu_estimate_noise_var_alone(ofdm, case):
    """lsmrc_estimate_noise_var on the same inputs: every frame's estimate within rtol 1e-5 of noise_var64 (the frames'
    noise levels all differ, so a frame-index error shows), bit-identical on a repeat call; constellation points on the
    kernel's fp32 levels give exactly 0"""
    import torch

    F, D, N, b = case
    K = N - 1
    y, E, _ = soft_inputs(F, D, N, b, seed=F * 1000 + D * 10 + b)
    rng = np.random.default_rng(F + D + N + b)
    af = np.float32(A_EXACT[b])
    levels = np.array([np.float32(k) * af for k in range(1, {2: 2, 4: 4, 6: 8}[b], 2)], np.float32)
    exact = levels[rng.integers(0, levels.size, (F, D, K, 2))] * np.where(rng.random((F, D, K, 2)) < 0.5, np.float32(-1), np.float32(1))
    exact = np.ascontiguousarray(exact).view(np.complex64)[..., 0]
    dev = torch.device("cuda:0")
    d_e = torch.from_numpy(E).to(dev)
    outs = [torch.full((F + 1,), float("nan"), device=dev) for _ in range(3)]
    torch.cuda.synchronize()
    with ofdm.LsMrcReceiver(1, N, 0, D + 1, b) as r:
        for x, o in zip((y, y, exact), outs):
            r.estimate_noise_var(torch.from_numpy(x).to(dev), d_e, F, o[:F])
            r.sync()
    got, again, zero = (o.cpu().numpy() for o in outs)
    assert np.isnan(got[F]) and np.isnan(zero[F])                              # (nothing past frame F - 1)
    want = noise_var64(y, E, b)
    assert np.all(np.abs(got[:F] - want) <= 1e-5 * want), (np.abs(got[:F] - want) / want).max()
    assert got.tobytes() == again.tobytes()
    assert (zero[:F] == 0).all(), zero[:F]


def _graph_case(ofdm, dims, policy, one_launch, want_fused):
    import torch

    A, N, C, S, b, F = dims
    K = N - 1
    dev = torch.device("cuda:0")
    user = torch.cuda.Stream(dev)
    g = torch.Generator(device=dev).manual_seed(13)
    inputs = [torch.randn((F, S, A, N + C, 2), device=dev, generator=g) for _ in range(3)]
    rx = torch.empty_like(inputs[0])
    comb = torch.zeros((F, S - 1, K, 2), device=dev)
    bits = torch.zeros((F, S - 1, (K * b + 7) // 8), device=dev, dtype=torch.uint8)
    llr = torch.zeros((F, S - 1, K, b), device=dev)
    outs = (comb, bits, llr)
    torch.cuda.synchronize(dev)
    with _receiver(ofdm, dims, ofdm.synth.make_pilot(K, 3), policy, one_launch) as r:
        r.set_stream(user.cuda_stream)

        def call(nv):
            r.demod_frames_device_soft(rx, F, comb, llr, nv, bits)

        with torch.cuda.stream(user):
            rx.copy_(inputs[0])
            call(0.25)                                     # first call: channel state allocated outside the capture
        user.synchronize()
        n_fused = r.one_launch_frames_count()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=user):
            call(0.25)
        for x in inputs:
            with torch.cuda.stream(user):
                rx.copy_(x)
                for o in outs:
                    o.zero_()
                graph.replay()
            user.synchronize()
            got = [o.clone() for o in outs]
            with torch.cuda.stream(user):
                for o in outs:
                    o.zero_()
                call(0.25)
            user.synchronize()
            assert all(torch.equal(a, o) for a, o in zip(got, outs))
            assert bool(torch.isfinite(llr).all()) and float(llr.abs().max()) > 0
        assert (r.one_launch_frames_count() > n_fused) == want_fused
        r.set_stream(None)


@pytest.mark.gpu
@pytest.mark.parametrize("which", ["frames_sh", "kernel_pair"])
def test_gpu_soft_call_replays_from_a_cuda_graph(ofdm, which):
    """the soft call on the caller's stream, captured once and replayed on three inputs: each replay equals an ordinary
    call (the LLR pointer and 1/noise_var are kernel arguments, nothing is kept on the host between calls)"""
    if which == "frames_sh":
        _graph_case(ofdm, (3, 2048, 144, 8, 4, 140), 2, True, True)
    else:
        _graph_case(ofdm, (16, 1024, 64, 6, 4, 7), 0, True, False)


@pytest.mark.gpu
def test_gpu_soft_and_hard_calls_interleave_on_one_handle(ofdm):
    """soft, hard, soft, hard on one handle, with batch sizes that take different kernels (single launch, one-launch
    kernel): each repeat is bit-identical to its first run, and a hard call writes no LLRs"""
    import torch

    A, N, C, S, b = 3, 2048, 144, 8, 4
    K = N - 1
    dev = torch.device("cuda:0")
    big, pilot = _frames(ofdm, (A, N, C, S, b, 140), seed=21, dev=dev)
    small = big[:2].contiguous()
    nv = _noise_var_of(N, b)
    llrs = {}

    def soft(r, rx, F):
        comb = torch.zeros((F, S - 1, K, 2), device=dev)
        bits = torch.zeros((F, S - 1, (K * b + 7) // 8), device=dev, dtype=torch.uint8)
        llr = llrs.setdefault(F, torch.empty((F, S - 1, K, b), device=dev))
        llr.zero_()
        torch.cuda.synchronize()
        r.demod_frames_device_soft(rx, F, comb, llr, nv, bits)
        r.sync()
        return [t.cpu().numpy() for t in (comb, bits, llr)]

    def hard(r, rx, F):
        comb = torch.zeros((F, S - 1, K, 2), device=dev)
        bits = torch.zeros((F, S - 1, (K * b + 7) // 8), device=dev, dtype=torch.uint8)
        torch.cuda.synchronize()
        r.demod_frames_device(rx, F, comb, bits)
        r.sync()
        return [t.cpu().numpy() for t in (comb, bits)]

    with _receiver(ofdm, (A, N, C, S, b, 140), pilot, 2, True) as r:
        s1 = soft(r, big, 140)
        h1 = hard(r, small, 2)
        s2 = soft(r, small, 2)
        h2 = hard(r, big, 140)
        s3 = soft(r, big, 140)
        h3 = hard(r, small, 2)
        s4 = soft(r, small, 2)
        for F, rx in ((2, small), (140, big)):      # hard calls after soft ones write nothing into the LLR buffers
            llrs[F].fill_(float("nan"))             # the last soft calls of either size used
            torch.cuda.synchronize()
            r.demod_frames_device(rx, F, torch.zeros((F, S - 1, K, 2), device=dev))
            r.sync()
            assert torch.isnan(llrs[F]).all(), F
        assert r.one_launch_frames_count() == 4 and r.oneshot_count() == 5
    for x, y in [(s1, s3), (s2, s4), (h1, h3)]:
        assert all(a.tobytes() == c.tobytes() for a, c in zip(x, y))
    assert s1[0].tobytes() == h2[0].tobytes() and s1[1].tobytes() == h2[1].tobytes()
    assert s2[0].tobytes() == h1[0].tobytes() and s2[1].tobytes() == h1[1].tobytes()


@pytest.mark.gpu
def test_gpu_soft_call_argument_errors(ofdm):
    """noise_var must be finite, > 0 and have a finite float reciprocal: 0, -1, NaN, +-inf and subnormals such as 1e-40
    (whose reciprocal overflows to inf, which would make the LLRs +-inf or NaN) are LSMRC_ERR_INVALID; the smallest
    normal float is accepted and gives finite LLRs"""
    import torch

    A, N, C, S, b, F = 4, 64, 16, 6, 2, 2
    K = N - 1
    dev = torch.device("cuda:0")
    rx, pilot = _frames(ofdm, (A, N, C, S, b, F), seed=5, dev=dev)
    rx = rx * 2.0 ** -20                 # (exact: |H|^2 ~ 1e-12, so that rho = sum|H|^2 / 1.18e-38 stays finite)
    comb = torch.zeros((F, S - 1, K, 2), device=dev)
    llr = torch.full((F, S - 1, K, b), float("nan"), device=dev)
    tiny = float(np.finfo(np.float32).tiny)
    torch.cuda.synchronize()
    with ofdm.LsMrcReceiver(A, N, C, S, b) as r:
        r.set_pilot(pilot)
        for nv in [0.0, -0.0, -1.0, float("nan"), float("inf"), float("-inf"), 1e-40, tiny / 8]:
            with pytest.raises(ofdm.LsmrcError) as e:
                r.demod_frames_device_soft(rx, F, comb, llr, nv)
            assert e.value.code == -1, nv                               # LSMRC_ERR_INVALID
        r.sync()
        assert torch.isnan(llr).all()                                   # nothing launched
        r.demod_frames_device_soft(rx, F, comb, llr, tiny)
        r.sync()
    got = llr.cpu().numpy()
    assert np.isfinite(got).all() and np.abs(got).max() > 1e20
    ref = ref_chain64(rx.cpu().numpy(), pilot, C, b, float(np.float32(tiny)))
    assert_llrs_within_bound(got, ref, b, "noise_var = FLT_MIN")
