"""User counts that leave the last user group of the multi-user data kernel partial, on every plan.

lsmrc_mu_data<PL, UG, SOFT> keeps the sums of UG users in registers and runs the row transforms once per group of UG
users (mu_ug in csrc/lsmrc_capi.cu: 8 users per pass at 64 points, 4 at 128 and 256, 2 at 1024 and 4096, 1 at 512 and
2048).  When UG does not divide U, the last group is padded up to UP = ceil(U / UG) * UG users: the padding users'
detector rows are zero, the detector rows of frame f start at f * UP, and the epilogue must store U users' rows and no
more -- teams of whole warps (1024, 4096 points) leave the group early, narrower teams (64..256) run the padding users'
epilogue without storing so that every lane reaches the same barriers.

Every case runs the hard and the soft call with time-orthogonal and with comb pilots.  Every output starts NaN- or
0xA5-filled and is followed by a guard tail; each (frame, user) row is compared on its own with the float64 reference
mu_ref64, so that one wrong user cannot hide behind the scale of the others."""
import numpy as np
import pytest

from mu_ref64 import mu_ref64, soft_ref
from test_multi_user_comb import comb_frames, llr_row_err, noise_var_of
from util import assert_bits_match

GUARD = 4096          # sentinel elements after every output buffer
BYTE_FILL = 0xA5
SNR = 25.0


def _row_rel_err(got, ref, axes):
    """largest |got - ref| over `axes` of each row, over that row's own largest |ref|"""
    d = np.abs(np.asarray(got).astype(np.complex128) - ref).max(axis=axes)
    return d / np.maximum(np.abs(ref).max(axis=axes), 1e-30)


def tolerances(ref):
    """(combined, soft) relative tolerance of the fp32 kernels against mu_ref64, as in the other multi-user tests"""
    return max(1e-5, 4e-6 * ref["gram_cond"]), max(2e-5, 4e-6 * ref["gram_cond"])


def check_rows(got, ref, want, b):
    """Every output of one multi-user call against the float64 reference, (frame, user) row by row; raises
    AssertionError naming the first bad row.  got: host arrays hconj [F,U,A,K], combined [F,D,U,K], bits [F,D,U,row]
    and, for the soft call, llr [F,D,U,K,b], sinr [F,U,K]; want: soft_ref of ref (or None)."""
    F, D, U, K = ref["combined"].shape
    tol, tol_s = tolerances(ref)
    for key in ("hconj", "combined", "llr", "sinr"):
        if key in got:
            bad = ~np.isfinite(np.ascontiguousarray(got[key]).view(np.float32))
            assert not bad.any(), f"{key}: {int(bad.sum())} elements not written or not finite, first at {np.argwhere(bad)[0]}"
    pad = got["bits"].shape[-1] * 8 - K * b                      # pack_bits leaves the bits after the last symbol zero
    last = got["bits"][..., -1] >> (8 - pad) if pad else np.zeros(1, np.uint8)
    assert not last.any(), f"bits: padding bits set in {int((last != 0).sum())} rows, first at {np.argwhere(last != 0)[0]}"
    checks = [("hconj", _row_rel_err(got["hconj"], ref["hconj"], (2, 3)), 1e-5),           # [F,U]
              ("combined", _row_rel_err(got["combined"], ref["combined"], (1, 3)), tol)]   # [F,U]
    if want is not None:
        checks += [("llr", llr_row_err(got["llr"], want["llr"]).max(axis=1), tol_s),       # [F,D,U] -> [F,U]
                   ("sinr", _row_rel_err(got["sinr"], want["sinr"], (2,)), tol_s)]
    for key, err, t in checks:
        assert err.shape == (F, U), (key, err.shape)
        f, u = np.unravel_index(int(np.argmax(err)), err.shape)
        assert err[f, u] <= t, f"{key}: (frame {f}, user {u}) off by {err[f, u]:.3e} of its own scale > {t:.3g}"
    for f in range(F):
        for u in range(U):
            assert_bits_match(got["bits"][f, :, u], ref["bits"][f, :, u], ref["combined"][f, :, u], b, f"bits (frame {f}, user {u})",
                              got["combined"][f, :, u], tol=tol)


# ------------------------------------------------------------------------------------------------ CPU
def _oracle_mu(*args, **kw):
    from test_multi_user import oracle_mu

    return oracle_mu(*args, **kw)


@pytest.mark.parametrize("b", [2, 4, 6])
def test_time_reference_single_user_is_the_single_user_chain(ofdm, b):
    """U = 1: ZF is MRC, inv(G) = 1 / sum|H|^2; combined and LLRs are those of the single-user float64 chain"""
    from test_soft_output import ref_chain64

    A, N, C, S, F = 8, 64, 16, 5, 2
    nv = noise_var_of(15.0, N)
    d = ofdm.synth.make_frames(F, A, N, C, S, b, snr_db=15.0, seed=80 + b)
    ref = mu_ref64(d["rx"], d["pilot_asc"], C, 1, 0.0, b)
    chain = ref_chain64(d["rx"], d["pilot_asc"], C, b, nv)
    assert ref["n_singular"] == 0
    assert np.abs(ref["combined"][:, :, 0] - chain["y"]).max() <= 1e-12 * np.abs(chain["y"]).max()
    assert np.abs(ref["ginv_diag"][:, 0] * chain["E"] - 1).max() <= 1e-12
    llr = soft_ref(ref, "zf", nv, b)["llr"][:, :, 0]
    assert np.abs(llr - chain["llr"]).max() <= 1e-12 * np.abs(chain["llr"]).max()
    # the time and comb frames are the same at U = 1, and so are the two branches of the reference
    c = ofdm.synth.make_frames_mu(F, A, N, C, S, b, 1, snr_db=15.0, seed=80 + b, pilots="comb")
    assert c["rx"].tobytes() == d["rx"].tobytes()
    comb = mu_ref64(d["rx"], d["pilot_asc"], C, 1, 0.0, b, pilots="comb")
    for key in ("hconj", "combined", "ginv_diag"):
        assert np.abs(comb[key] - ref[key]).max() <= 1e-13 * np.abs(ref[key]).max(), key
    assert np.array_equal(comb["bits"], ref["bits"])


@pytest.mark.parametrize("U,A,N", [(3, 8, 64), (5, 12, 256), (9, 24, 64)])
def test_time_reference_recovers_noiseless_constellation(ofdm, U, A, N):
    C, S, b, F = N // 8, U + 3, 4, 2
    d = ofdm.synth.make_frames_mu(F, A, N, C, S, b, U, snr_db=None, seed=200 + U)
    ref = mu_ref64(d["rx"], d["pilot_asc"], C, U, 0.0, b)
    assert ref["n_singular"] == 0 and ref["combined"].shape == (F, S - U, U, N - 1)
    sent = ofdm.synth.qam_map_indices(d["src_idx"], b)
    # (the frames are complex64: the estimate carries their rounding)
    assert _row_rel_err(np.conj(ref["hconj"]), d["h_true"].astype(np.complex128), (2, 3)).max() <= 1e-6
    assert _row_rel_err(ref["combined"], sent, (1, 3)).max() <= 1e-6 * ref["gram_cond"]
    assert np.array_equal(ref["bits"], ofdm.synth.pack_bits_rows(d["src_idx"], b))


@pytest.mark.parametrize("detector", ["zf", "mmse"])
@pytest.mark.parametrize("U,A,N", [(5, 12, 64), (7, 16, 256)])
def test_time_reference_matches_the_c_oracle(ofdm, U, A, N, detector):
    """the C oracle (fp32 LS estimate and FFT, float64 detector) within its fp32 tolerance, with odd U"""
    C, S, b, F = N // 8, U + 2, 4, 3
    lam = 0.05 if detector == "mmse" else 0.0
    d = ofdm.synth.make_frames_mu(F, A, N, C, S, b, U, snr_db=20.0, seed=300 + U)
    ref = mu_ref64(d["rx"], d["pilot_asc"], C, U, lam, b)
    got = _oracle_mu(d["rx"], d["pilot_asc"], C, U, b, lam)
    assert ref["n_singular"] == got["n_singular"] == 0
    tol, _ = tolerances(ref)
    assert _row_rel_err(got["hconj"], ref["hconj"], (2, 3)).max() <= 1e-5
    assert _row_rel_err(got["combined"], ref["combined"], (1, 3)).max() <= tol
    for u in range(U):
        assert_bits_match(got["bits"][:, :, u], ref["bits"][:, :, u], ref["combined"][:, :, u], b, "bits", got["combined"][:, :, u], tol=tol)


@pytest.fixture(scope="module")
def comparator_case(ofdm):
    """a time-pilot soft call's worth of reference outputs, rounded to the kernels' types (U = 5, F = 3)"""
    A, N, C, U, b, F = 12, 64, 16, 5, 4, 3
    nv = noise_var_of(SNR, N)
    d = ofdm.synth.make_frames_mu(F, A, N, C, U + 2, b, U, snr_db=SNR, seed=7)
    ref = mu_ref64(d["rx"], d["pilot_asc"], C, U, 0.0, b)
    want = soft_ref(ref, "zf", nv, b)
    got = {"hconj": ref["hconj"], "combined": ref["combined"], "bits": ref["bits"], "llr": want["llr"], "sinr": want["sinr"]}
    got = {k: np.ascontiguousarray(v, np.uint8 if k == "bits" else np.float32 if k in ("llr", "sinr") else np.complex64)
           for k, v in got.items()}
    return ref, want, got, b


USER_AXIS = {"hconj": 1, "combined": 2, "bits": 2, "llr": 2, "sinr": 1}
MUTATIONS = [(m, key) for m in ("last_user_zeroed", "last_user_is_user_U-2", "frame_1_shifted_by_one_user") for key in USER_AXIS] + \
    [("one_element_nan", key) for key in ("hconj", "combined", "llr", "sinr")] + [("padding_bit_set", "bits")]


def test_comparator_accepts_the_rounded_reference(comparator_case):
    ref, want, got, b = comparator_case
    check_rows(got, ref, want, b)


@pytest.mark.parametrize("mutation,key", MUTATIONS)
def test_comparator_rejects_plausible_kernel_mistakes(comparator_case, mutation, key):
    """the mistakes of a kernel that gets the padded last user group wrong: a row never stored (zeros, or whatever the
    buffer held), a row of the wrong user, frame f's rows at f * UP instead of f * U (or the reverse), a store skipped"""
    ref, want, got, b = comparator_case
    bad = {k: v.copy() for k, v in got.items()}
    x = bad[key]
    ax = USER_AXIS[key]
    U = x.shape[ax]
    last, other = [slice(None)] * x.ndim, [slice(None)] * x.ndim
    last[ax], other[ax] = U - 1, U - 2
    if mutation == "last_user_zeroed":
        x[tuple(last)] = 0
    elif mutation == "last_user_is_user_U-2":
        x[tuple(last)] = x[tuple(other)]
    elif mutation == "frame_1_shifted_by_one_user":
        x[1] = np.roll(x[1], 1, axis=ax - 1)
    elif mutation == "one_element_nan":
        x.view(np.float32).reshape(-1)[x.view(np.float32).size // 2 + 1] = np.nan
    else:
        x[2, 1, U - 1, -1] |= 0x80
    with pytest.raises(AssertionError):
        check_rows(bad, ref, want, b)


# ------------------------------------------------------------------------------------------------ GPU
# (A, N, C, U, b, detector, S with time pilots, S with comb pilots); A >= 2U keeps the Gram matrices well conditioned.
# The time cases run the listed detector, the comb cases the other one.  For each plan: U < UG (one partial group),
# U > UG with U % UG != 0 (several groups, the last partial; with S = U + 1 on one case per narrow plan, one data symbol:
# neighbouring teams of a warp hold different groups), and U = 7, 5 at the UG = 1 plans as controls.
CASES = [
    (8, 64, 16, 3, 4, "zf", 5, 3),
    (24, 64, 16, 9, 2, "mmse", 10, 4),
    (32, 64, 16, 15, 4, "zf", 17, 5),
    (8, 128, 16, 3, 6, "mmse", 5, 3),
    (12, 128, 16, 5, 4, "zf", 7, 4),
    (24, 128, 16, 11, 2, "mmse", 12, 5),
    (8, 256, 32, 3, 2, "zf", 5, 5),
    (12, 256, 32, 6, 4, "mmse", 8, 3),
    (28, 256, 32, 13, 6, "zf", 14, 4),
    (16, 512, 32, 7, 4, "mmse", 9, 4),
    (4, 1024, 64, 1, 4, "mmse", 3, 3),
    (8, 1024, 64, 3, 6, "zf", 5, 3),
    (12, 1024, 64, 5, 4, "mmse", 7, 5),
    (32, 1024, 64, 15, 2, "zf", 17, 4),
    (12, 2048, 144, 5, 4, "zf", 7, 3),
    (4, 4096, 288, 1, 2, "zf", 3, 4),
    (8, 4096, 288, 3, 4, "mmse", 5, 4),
    (20, 4096, 288, 9, 6, "zf", 11, 3),
]
_CASE_ID = "A{}_N{}_C{}_U{}_b{}_{}_St{}_Sc{}"
F = 3                 # the per-frame stride of the detector rows is crossed twice


def _guarded(n, dtype, fill, dev):
    import torch

    return torch.full((n + GUARD,), fill, dtype=dtype, device=dev)


def _call(r, d_rx, U, b, detector, nv, soft, P):
    """one multi-user call on guarded, filled outputs -> dict of host arrays; asserts that no guard tail was touched"""
    import torch

    A, N, S = r.cfg.n_ant, r.cfg.fft_size, r.cfg.n_sym
    K, D = N - 1, S - P
    row = (K * b + 7) // 8
    dev = torch.device("cuda:0")
    nan = float("nan")
    shapes = {"combined": (F, D, U, K, 2), "bits": (F, D, U, row), "hconj": (F, U, A, K, 2)}
    if soft:
        shapes.update(llr=(F, D, U, K, b), sinr=(F, U, K))
    bufs, outs = {}, {}
    for key, shape in shapes.items():
        n = int(np.prod(shape))
        bufs[key] = _guarded(n, torch.uint8, BYTE_FILL, dev) if key == "bits" else _guarded(n, torch.float32, nan, dev)
        outs[key] = bufs[key][:n]
    torch.cuda.synchronize()
    if soft:
        bad = r.demod_frames_device_mu_soft(d_rx, F, U, outs["combined"], outs["llr"], outs["bits"], outs["hconj"], outs["sinr"],
                                            detector=detector, noise_var=nv, count_singular=True)
    else:
        bad = r.demod_frames_device_mu(d_rx, F, U, outs["combined"], outs["bits"], outs["hconj"], detector=detector, noise_var=nv,
                                       count_singular=True)
    r.sync()
    got = {"n_singular": bad}
    for key, shape in shapes.items():
        n = outs[key].numel()
        tail = bufs[key][n:].cpu().numpy()
        assert (tail == BYTE_FILL).all() if key == "bits" else (tail.view(np.uint32) == 0x7FC00000).all(), f"{key}: write past the end"
        host = outs[key].cpu().numpy().reshape(shape)
        got[key] = host.view(np.complex64)[..., 0] if key in ("combined", "hconj") else host
    return got


def _run_layout(ofdm, case, pilots):
    """hard and soft call of one layout against mu_ref64: (reference, hard, soft)"""
    import torch

    A, N, C, U, b, det, S_time, S_comb = case
    if pilots == "comb":
        det = "mmse" if det == "zf" else "zf"
    nv = noise_var_of(SNR, N)
    lam = nv if det == "mmse" else 0.0
    seed = N + 17 * U + (1 if pilots == "comb" else 0)
    if pilots == "time":
        S, P = S_time, U
        d = ofdm.synth.make_frames_mu(F, A, N, C, S, b, U, snr_db=SNR, seed=seed)
    else:
        S, P = S_comb, 1
        d = comb_frames(F, A, N, C, S, b, U, SNR, seed)
    ref = mu_ref64(d["rx"], d["pilot_asc"], C, U, lam, b, pilots=pilots)
    assert ref["n_singular"] == 0
    want = soft_ref(ref, det, nv, b)
    with ofdm.LsMrcReceiver(A, N, C, S, b) as r:
        r.set_pilot(d["pilot_asc"])
        r.set_mu_pilots(pilots)
        d_rx = torch.from_numpy(d["rx"]).to("cuda:0")
        hard = _call(r, d_rx, U, b, det, nv, False, P)
        soft = _call(r, d_rx, U, b, det, nv, True, P)
    return ref, want, hard, soft


@pytest.mark.gpu
@pytest.mark.parametrize("pilots", ["time", "comb"])
@pytest.mark.parametrize("case", CASES, ids=lambda c: _CASE_ID.format(*c))
def test_gpu_partial_user_groups(ofdm, case, pilots):
    """hard and soft call: every element written and finite, no guard tail touched, the bits rows' padding zero, each
    (frame, user) row of hconj / combined / bits / LLR / SINR within the fp32 tolerance of mu_ref64, and the soft call's
    combined, bits and hconj byte-identical to the hard call's"""
    ref, want, hard, soft = _run_layout(ofdm, case, pilots)
    assert hard["n_singular"] == soft["n_singular"] == 0
    check_rows(hard, ref, None, case[4])
    check_rows(soft, ref, want, case[4])
    for key in ("combined", "bits", "hconj"):
        assert soft[key].tobytes() == hard[key].tobytes(), key


def _mu_data_launches(fn):
    """(N, UG, soft) of every lsmrc_mu_data launch of fn(), from torch.profiler"""
    import re

    from test_soft_output import _kernel_launches

    out = set()
    for name, _ in _kernel_launches(fn):
        m = re.search(r"lsmrc_mu_data<lsmrc::Plan<(?:\(int\))?(\d+),[^>]*>, (?:\(int\))?(\d+), (?:\(bool\))?(true|false|1|0)>", name)
        if m:
            out.add((int(m.group(1)), int(m.group(2)), m.group(3) in ("true", "1")))
    return out


def launched_mu_data():
    """{N: sorted (UG, soft) launched} for the hard and the soft call of the first CASES entry of each plan"""
    import ofdm_b200
    import torch

    seen = {}
    for N in (64, 128, 256, 512, 1024, 2048, 4096):
        A, _, C, U, b, det, S, _ = next(c for c in CASES if c[1] == N)
        nv = noise_var_of(SNR, N)
        d = ofdm_b200.synth.make_frames_mu(1, A, N, C, S, b, U, snr_db=SNR, seed=N)
        d_rx = torch.from_numpy(d["rx"]).to("cuda:0")
        K = N - 1
        comb = torch.empty((1, S - U, U, K, 2), device="cuda:0")
        llr = torch.empty((1, S - U, U, K, b), device="cuda:0")
        with ofdm_b200.LsMrcReceiver(A, N, C, S, b) as r:
            r.set_pilot(d["pilot_asc"])

            def call():
                r.demod_frames_device_mu(d_rx, 1, U, comb, detector=det, noise_var=nv)
                r.demod_frames_device_mu_soft(d_rx, 1, U, comb, llr, detector=det, noise_var=nv)
                r.sync()

            call()                                       # (first calls: scratch allocated)
            seen[N] = sorted(_mu_data_launches(call))
    return seen


# The profiling runs in a child process.  Run in the pytest process, a torch.profiler session here followed by the GPU
# tests of test_multi_user_soft.py leaves that process unable to record kernels: test_soft_output's route map, profiled
# later in the same process, then sees no kernel launch at all (B200, torch 2.11; without the earlier session, or
# without those tests in between, it sees them).
_CHILD = """
import json, os, sys
sys.path[:0] = [sys.argv[1], os.path.join(sys.argv[1], "tests")]
import test_multi_user_groups
print(json.dumps(test_multi_user_groups.launched_mu_data()))
"""


@pytest.mark.gpu
def test_gpu_route_map():
    """reads UG from the launched lsmrc_mu_data<Plan, UG, SOFT> of each plan and checks that CASES still covers, per
    plan, a single partial group (U < UG) and several groups with the last one partial (U > UG, U % UG != 0) -- or,
    at UG = 1, has a control case -- so that retuning mu_ug cannot quietly take the padding out of the sweep"""
    import json
    import os
    import subprocess
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    flags = ["-B"] + (["-s"] if sys.flags.no_user_site else [])
    r = subprocess.run([sys.executable, *flags, "-c", _CHILD, root], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-4000:]
    launched = {int(n): v for n, v in json.loads(r.stdout.strip().splitlines()[-1]).items()}
    table = []
    for N in (64, 128, 256, 512, 1024, 2048, 4096):
        seen = launched[N]
        assert {n for n, _, _ in seen} == {N} and {s for _, _, s in seen} == {False, True}, (N, seen)
        ugs = {ug for _, ug, _ in seen}
        assert len(ugs) == 1, (N, seen)
        ug = ugs.pop()
        users = sorted(c[3] for c in CASES if c[1] == N)
        single = [u for u in users if u < ug]
        several = [u for u in users if u > ug and u % ug]
        table.append(f"N={N:5d} UG={ug}  U in CASES {users}  one partial group {single}  several, last partial {several}")
        if ug > 1:
            assert single and several, table[-1]
        else:
            assert users, table[-1]
    print("\n".join(table))


@pytest.mark.gpu
@pytest.mark.parametrize("A,N,C,U", [(24, 64, 16, 11), (16, 256, 32, 7), (12, 1024, 64, 5), (8, 4096, 288, 3)])
def test_gpu_singular_subcarriers_at_odd_user_counts(ofdm, A, N, C, U):
    """Users U-2 and U-1 (both in the padded last group at 64 and 256 points) share a channel on a few subcarriers:
    those are exact zeros for every user in combined, LLRs and SINR, their count is the reference's, and every other
    subcarrier matches the reference"""
    import torch

    b, S, nv = 4, U + 2, 1e-3
    K = N - 1
    rng = np.random.default_rng(U)
    h = (rng.standard_normal((F, U, A, K)) + 1j * rng.standard_normal((F, U, A, K))) / np.sqrt(2.0)
    ks = [0, 17, K // 2, K - 1]                  # subcarrier index k = bin - 1
    h[:, U - 1][:, :, ks] = h[:, U - 2][:, :, ks]
    d = ofdm.synth.make_frames_mu(F, A, N, C, S, b, U, snr_db=None, seed=U, h=h)
    ref = mu_ref64(d["rx"], d["pilot_asc"], C, U, 0.0, b)
    assert ref["n_singular"] == F * len(ks)
    want = soft_ref(ref, "zf", nv, b)
    pos = [k + N // 2 if k + 1 < N // 2 else k + 1 - N // 2 for k in ks]          # ascending-frequency index of bin k + 1
    with ofdm.LsMrcReceiver(A, N, C, S, b) as r:
        r.set_pilot(d["pilot_asc"])
        d_rx = torch.from_numpy(d["rx"]).to("cuda:0")
        hard = _call(r, d_rx, U, b, "zf", nv, False, U)
        soft = _call(r, d_rx, U, b, "zf", nv, True, U)
    for got in (hard, soft):
        assert got["n_singular"] == ref["n_singular"]
        assert (got["combined"][..., pos] == 0).all()
        check_rows(got, ref, want if got is soft else None, b)
    assert (soft["llr"][..., pos, :] == 0).all() and (soft["sinr"][..., pos] == 0).all()
    rest = np.setdiff1d(np.arange(K), pos)
    assert (soft["sinr"][..., rest] > 0).all()
