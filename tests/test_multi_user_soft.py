"""Multi-user uplink with soft output (lsmrc_demod_frames_device_mu_soft): per-user post-detection SINR and max-log
LLRs of the ZF / MMSE detector (DESIGN.md 8f).  The CPU oracle is oracle_mu_soft in tests/cpp/mu_soft_oracle.c (which
includes the hard oracle tests/cpp/mu_oracle.c): it starts from the hconj and combined of oracle_demod_frames_mu and
reuses the single-user oracle's LLR formula.  It is built here into a temporary directory."""
import ctypes
import os
import shutil
import subprocess
import tempfile

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_LIB = {}


def _mu_lib():
    if "lib" not in _LIB:
        d = tempfile.mkdtemp(prefix="mu_soft_oracle_")
        so = os.path.join(d, "libmu_oracle.so")
        srcs = [os.path.join(ROOT, "tests", "cpp", "mu_soft_oracle.c"), os.path.join(ROOT, "oracle", "cpuls_oracle.c"),
                os.path.join(ROOT, "oracle", "fft_shim.c")]
        subprocess.run([os.environ.get("CC", "gcc"), "-O2", "-fPIC", "-ffp-contract=off", "-pthread", "-shared", "-o", so, *srcs,
                        "-lm"], check=True)
        lib = ctypes.CDLL(so)
        shutil.rmtree(d, ignore_errors=True)  # (the mapping stays valid)
        lib.oracle_demod_frames_mu.restype = ctypes.c_int
        lib.oracle_demod_frames_mu.argtypes = [ctypes.c_void_p, ctypes.c_void_p] + [ctypes.c_int] * 7 + [ctypes.c_double] + \
            [ctypes.c_void_p] * 3
        lib.oracle_mu_soft.restype = ctypes.c_int
        lib.oracle_mu_soft.argtypes = [ctypes.c_void_p, ctypes.c_void_p] + [ctypes.c_int] * 6 + [ctypes.c_double] * 2 + \
            [ctypes.c_void_p] * 2
        _LIB["lib"] = lib
    return _LIB["lib"]


def noise_var_of(snr_db, N):
    """noise variance per antenna and subcarrier after the FFT of synth.make_frames_mu's AWGN at snr_db"""
    return (N - 1) / N * 10.0 ** (-snr_db / 10.0)


def oracle_mu_soft(rx, pilot_asc, cp, n_users, qam_bits, detector, noise_var):
    """rx [F,S,A,N+C] -> dict(hconj [F,U,A,K], combined [F,S-U,U,K], bits [F,S-U,U,row], sinr [F,U,K] float64,
    llr [F,S-U,U,K,b] float32, n_singular).  MMSE loads the diagonal with lambda = noise_var."""
    rx = np.ascontiguousarray(rx, np.complex64)
    F, S, A, NC = rx.shape
    N = NC - cp
    K, U = N - 1, n_users
    lam = noise_var if detector == "mmse" else 0.0
    pilot_asc = np.ascontiguousarray(pilot_asc, np.complex64)
    hconj = np.empty((F, U, A, K), np.complex64)
    comb = np.empty((F, S - U, U, K), np.complex64)
    bits = np.zeros((F, S - U, U, (K * qam_bits + 7) // 8), np.uint8)
    lib = _mu_lib()
    bad = lib.oracle_demod_frames_mu(rx.ctypes.data, pilot_asc.ctypes.data, F, S, A, N, cp, U, qam_bits, float(lam),
                                     hconj.ctypes.data, comb.ctypes.data, bits.ctypes.data)
    sinr = np.empty((F, U, K), np.float64)
    llr = np.empty((F, S - U, U, K, qam_bits), np.float32)
    bad2 = lib.oracle_mu_soft(hconj.ctypes.data, comb.ctypes.data, F, S, N, A, U, qam_bits, float(lam), float(noise_var),
                              sinr.ctypes.data, llr.ctypes.data)
    assert bad2 == bad
    return {"hconj": hconj, "combined": comb, "bits": bits, "sinr": sinr, "llr": llr, "n_singular": bad}


def gram_cond(hconj, noise_var=0.0):
    """largest condition number of G_k = H^H H + lambda I over frames and subcarriers; hconj [F,U,A,K]"""
    h = np.conj(hconj.astype(np.complex128)).transpose(0, 3, 2, 1)  # [F,K,A,U]
    g = np.conj(np.swapaxes(h, -1, -2)) @ h + noise_var * np.eye(h.shape[-1])
    return float(np.linalg.cond(g).max())


def bin_to_asc_pos(bin_idx, N):
    return bin_idx - 1 + N // 2 if bin_idx < N // 2 else bin_idx - N // 2


def unpack(bits, K, b):
    """packed rows [..., row] -> bits [..., K, b] (bit q of symbol i at position i*b + q, LSB first)"""
    return np.unpackbits(bits, axis=-1, bitorder="little")[..., : K * b].reshape(*bits.shape[:-1], K, b)


def llr_row_err(got, ref):
    """largest |got - ref| of each LLR row (last two axes [K, b]) over that row's max |ref|"""
    d = np.abs(got.astype(np.float64) - ref.astype(np.float64)).max(axis=(-1, -2))
    return d / np.maximum(np.abs(ref.astype(np.float64)).max(axis=(-1, -2)), 1e-30)


# ------------------------------------------------------------------------------------------------ CPU
@pytest.mark.parametrize("detector", ["zf", "mmse"])
@pytest.mark.parametrize("b", [2, 4, 6])
def test_oracle_single_user_is_the_single_user_soft_path(ofdm, oracle, detector, b):
    A, N, C, S, F, snr = 8, 64, 16, 6, 2, 18.0
    nv = noise_var_of(snr, N)
    d = ofdm.synth.make_frames(F, A, N, C, S, b, snr_db=snr, seed=21 + b)
    ref = oracle.demod_frames(d["rx"], d["pilot_asc"], b, C)
    want = oracle.soft_demap(ref["combined"], ref["hsqrd"], b, nv)       # [F,S-1,K,b]
    got = oracle_mu_soft(d["rx"], d["pilot_asc"], C, 1, b, detector, nv)
    assert got["n_singular"] == 0
    assert llr_row_err(got["llr"][:, :, 0], want).max() <= 1e-5
    rho = ofdm.synth.bin_to_asc(ref["hsqrd"].astype(np.float64)) / nv   # sum|H|^2 / sigma^2
    assert np.abs(got["sinr"][:, 0] - rho).max() <= 1e-5 * rho.max()


def _numpy_sinr(hconj, lam, sigma2):
    """SINR of every (frame, user, subcarrier) from W = inv(H^H H + lam I) H^H in float64, ascending frequency [F,U,K]:
    |[WH]_uu|^2 / (sum_{v != u} |[WH]_uv|^2 + sigma2 ||w_u||^2)"""
    from gpu_accel_ofdm_ls_mrc_b200.synth import bin_to_asc

    H = np.conj(hconj.astype(np.complex128)).transpose(0, 3, 2, 1)     # [F,K,A,U]
    Hh = np.conj(np.swapaxes(H, -1, -2))
    U = H.shape[-1]
    W = np.linalg.solve(Hh @ H + lam * np.eye(U), Hh)                  # [F,K,U,A]
    WH = W @ H
    p = np.abs(WH) ** 2
    sig = np.diagonal(p, axis1=-2, axis2=-1)
    interf = p.sum(-1) - sig
    wn = (np.abs(W) ** 2).sum(-1)
    return bin_to_asc((sig / (interf + sigma2 * wn)).transpose(0, 2, 1))


@pytest.mark.parametrize("U,A", [(2, 8), (4, 8), (8, 16)])
@pytest.mark.parametrize("detector", ["zf", "mmse"])
def test_oracle_sinr_from_first_principles(ofdm, U, A, detector):
    N, C, S, b, F, snr = 64, 16, U + 2, 4, 2, 15.0
    nv = noise_var_of(snr, N)
    d = ofdm.synth.make_frames_mu(F, A, N, C, S, b, U, snr_db=snr, seed=50 + U)
    got = oracle_mu_soft(d["rx"], d["pilot_asc"], C, U, b, detector, nv)
    assert got["n_singular"] == 0
    lam = nv if detector == "mmse" else 0.0
    kappa = gram_cond(got["hconj"], lam)
    want = _numpy_sinr(got["hconj"], lam, nv)
    rho = got["sinr"]
    assert (rho > 0).all()
    assert (np.abs(rho - want) <= 1e-9 * kappa * (rho + 1.0)).all(), (np.abs(rho - want) / (rho + 1)).max() / kappa


@pytest.mark.parametrize("detector", ["zf", "mmse"])
@pytest.mark.parametrize("b", [4, 6])
def test_oracle_llr_signs_are_the_hard_bits(ofdm, detector, b):
    U, A, N, C, S, F, snr = 4, 8, 64, 16, 8, 2, 12.0
    K = N - 1
    nv = noise_var_of(snr, N)
    d = ofdm.synth.make_frames_mu(F, A, N, C, S, b, U, snr_db=snr, seed=70 + b)
    got = oracle_mu_soft(d["rx"], d["pilot_asc"], C, U, b, detector, nv)
    hard = unpack(got["bits"], K, b)
    dec = (got["llr"] < 0).astype(np.uint8)
    assert np.array_equal(dec[..., :2], hard[..., :2])             # sign bits everywhere
    if detector == "zf":                                           # ZF: the LLRs are of the hard symbols themselves
        big = np.abs(got["llr"]) > 1e-6 * np.abs(got["llr"]).max()
        assert np.array_equal(dec[big], hard[big])
    else:                                                          # MMSE: the amplitude bits see the unbiased symbol
        assert not np.array_equal(dec, hard)


@pytest.mark.parametrize("detector", ["zf", "mmse"])
def test_oracle_llr_magnitude_ranks_reliability(ofdm, detector):
    """Bits with larger |LLR| are wrong less often: the bit error rate against the sent bits falls monotonically over
    five |LLR| quantile bins (U = 4 on A = 8, 16-QAM, 10 dB: about 3 % of the bits are wrong)."""
    U, A, N, C, S, b, F, snr = 4, 8, 256, 32, 12, 4, 6, 10.0
    K = N - 1
    nv = noise_var_of(snr, N)
    d = ofdm.synth.make_frames_mu(F, A, N, C, S, b, U, snr_db=snr, seed=123)
    got = oracle_mu_soft(d["rx"], d["pilot_asc"], C, U, b, detector, nv)
    sent = unpack(ofdm.synth.pack_bits_rows(d["src_idx"], b), K, b).ravel()
    llr = got["llr"].ravel().astype(np.float64)
    err = (llr < 0).astype(np.uint8) != sent
    assert 0.005 < err.mean() < 0.2, err.mean()
    edges = np.quantile(np.abs(llr), np.linspace(0.0, 1.0, 6))
    which = np.clip(np.searchsorted(edges, np.abs(llr), side="right") - 1, 0, 4)
    ber = [err[which == i].mean() for i in range(5)]
    assert all(ber[i] > ber[i + 1] for i in range(4)), ber


def test_oracle_mmse_unbiased_decisions_beat_the_biased_hard_bits(ofdm):
    """MMSE shrinks its output by beta = [WH]_uu < 1, so the hard demapper of lsmrc_demod_frames_device_mu decides the
    inner 16-QAM amplitude too often; the LLRs see x^ / beta.  At U = 4 on A = 8, 16-QAM, 16 dB, seed 321 (195840 bits,
    0.75 % wrong in the hard bits) the two disagree on 85 amplitude bits and the LLR sign is right on 58 of them:
    1430 bit errors instead of 1461."""
    U, A, N, C, S, b, F, snr = 4, 8, 256, 32, 10, 4, 8, 16.0
    K = N - 1
    nv = noise_var_of(snr, N)
    d = ofdm.synth.make_frames_mu(F, A, N, C, S, b, U, snr_db=snr, seed=321)
    got = oracle_mu_soft(d["rx"], d["pilot_asc"], C, U, b, "mmse", nv)
    sent = unpack(ofdm.synth.pack_bits_rows(d["src_idx"], b), K, b)
    soft = (got["llr"] < 0).astype(np.uint8)
    hard = unpack(got["bits"], K, b)
    differ = soft != hard
    assert not differ[..., :2].any() and differ.sum() >= 50
    assert (soft[differ] == sent[differ]).mean() >= 0.6
    assert (soft != sent).mean() <= (hard != sent).mean()


def test_abi_exports_the_soft_multi_user_entry_point(ofdm):
    lib = ofdm.load_library()
    assert "lsmrc_demod_frames_device_mu_soft" in ofdm.ABI
    assert hasattr(lib, "lsmrc_demod_frames_device_mu_soft")


# ------------------------------------------------------------------------------------------------ GPU
def _run_soft(ofdm, r, rx, F, U, b, detector, noise_var, want_hconj=True, want_sinr=True, count=False):
    import torch

    A, N, S = r.cfg.n_ant, r.cfg.fft_size, r.cfg.n_sym
    K = N - 1
    dev = torch.device("cuda:0")
    d_rx = torch.from_numpy(np.ascontiguousarray(rx)).to(dev) if isinstance(rx, np.ndarray) else rx
    nan = float("nan")                      # every output element is written: nothing may be left as filled
    comb = torch.view_as_complex(torch.full((F, S - U, U, K, 2), nan, device=dev))
    bits = torch.full((F, S - U, U, (K * b + 7) // 8), 0xA5, dtype=torch.uint8, device=dev)
    llr = torch.full((F, S - U, U, K, b), nan, device=dev)
    sinr = torch.full((F, U, K), nan, device=dev) if want_sinr else None
    hc = torch.view_as_complex(torch.full((F, U, A, K, 2), nan, device=dev)) if want_hconj else None
    torch.cuda.synchronize()
    bad = r.demod_frames_device_mu_soft(d_rx, F, U, comb, llr, bits, hc, sinr, detector=detector, noise_var=noise_var,
                                        count_singular=count)
    r.sync()
    return {"combined": comb.cpu().numpy(), "bits": bits.cpu().numpy(), "llr": llr.cpu().numpy(),
            "sinr": sinr.cpu().numpy() if want_sinr else None, "hconj": hc.cpu().numpy() if want_hconj else None,
            "n_singular": bad}


def _run_hard(ofdm, r, rx, F, U, b, detector, noise_var):
    import torch

    N, S = r.cfg.fft_size, r.cfg.n_sym
    K = N - 1
    dev = torch.device("cuda:0")
    d_rx = torch.from_numpy(np.ascontiguousarray(rx)).to(dev) if isinstance(rx, np.ndarray) else rx
    comb = torch.view_as_complex(torch.full((F, S - U, U, K, 2), float("nan"), device=dev))
    bits = torch.full((F, S - U, U, (K * b + 7) // 8), 0xA5, dtype=torch.uint8, device=dev)
    torch.cuda.synchronize()
    r.demod_frames_device_mu(d_rx, F, U, comb, bits, detector=detector, noise_var=noise_var)
    r.sync()
    return {"combined": comb.cpu().numpy(), "bits": bits.cpu().numpy()}


MU_CASES = [  # (A, N, C, S, U, detector, b) -- the shapes of test_multi_user.py, one per plan from 64 to 4096 points
    (4, 64, 16, 16, 2, "zf", 2),
    (16, 64, 16, 16, 4, "mmse", 2),
    (8, 128, 16, 10, 2, "zf", 4),
    (32, 256, 32, 12, 4, "zf", 4),
    (32, 512, 32, 12, 4, "mmse", 4),
    (64, 1024, 64, 20, 4, "zf", 4),
    (64, 1024, 64, 20, 8, "mmse", 4),
    (128, 2048, 144, 14, 8, "zf", 4),
    (256, 4096, 288, 14, 4, "zf", 6),
    (256, 4096, 288, 18, 16, "mmse", 6),  # (16 users need S > 16: 16 pilot symbols)
]


@pytest.mark.gpu
@pytest.mark.parametrize("case", MU_CASES, ids=lambda c: "A{}_N{}_C{}_S{}_U{}_{}_b{}".format(*c))
def test_gpu_soft_matches_oracle(ofdm, case):
    A, N, C, S, U, det, b = case
    F, snr = (2 if N >= 2048 else 3), 20.0
    nv = noise_var_of(snr, N)
    d = ofdm.synth.make_frames_mu(F, A, N, C, S, b, U, snr_db=snr, seed=A + N + U)
    ref = oracle_mu_soft(d["rx"], d["pilot_asc"], C, U, b, det, nv)
    assert ref["n_singular"] == 0
    with ofdm.LsMrcReceiver(A, N, C, S, b) as r:
        r.set_pilot(d["pilot_asc"])
        got = _run_soft(ofdm, r, d["rx"], F, U, b, det, nv, count=True)
    assert got["n_singular"] == 0
    kappa = gram_cond(ref["hconj"], nv if det == "mmse" else 0.0)
    tol = max(2e-5, 4e-6 * kappa)
    assert np.isfinite(got["llr"]).all() and np.isfinite(got["sinr"]).all()
    err = llr_row_err(got["llr"], ref["llr"])
    assert err.max() <= tol, (err.max(), tol, kappa)
    s_err = np.abs(got["sinr"] - ref["sinr"]).max(-1) / ref["sinr"].max(-1)
    assert s_err.max() <= tol, (s_err.max(), tol, kappa)


@pytest.mark.gpu
@pytest.mark.parametrize("detector", ["zf", "mmse"])
@pytest.mark.parametrize("dims", [(32, 1024, 64, 9, 5, 4), (16, 2048, 144, 8, 3, 4), (16, 64, 16, 12, 9, 2)],
                         ids=["N1024_U5", "N2048_U3", "N64_U9"])
def test_gpu_combined_and_bits_are_those_of_the_hard_call(ofdm, detector, dims):
    """U above the plan's users per pass (2 at 1024, 1 at 2048, 8 at 64 points): several user groups"""
    A, N, C, S, U, b = dims
    F = 3
    nv = noise_var_of(20.0, N)
    d = ofdm.synth.make_frames_mu(F, A, N, C, S, b, U, snr_db=20.0, seed=N + U)
    with ofdm.LsMrcReceiver(A, N, C, S, b) as r:
        r.set_pilot(d["pilot_asc"])
        soft = _run_soft(ofdm, r, d["rx"], F, U, b, detector, nv)
        hard = _run_hard(ofdm, r, d["rx"], F, U, b, detector, nv)
    assert soft["combined"].tobytes() == hard["combined"].tobytes()
    assert soft["bits"].tobytes() == hard["bits"].tobytes()
    assert (soft["llr"] != 0).any()


@pytest.mark.gpu
@pytest.mark.parametrize("detector", ["zf", "mmse"])
@pytest.mark.parametrize("dims", [(4, 64, 16, 16, 2), (16, 1024, 64, 6, 4), (16, 4096, 288, 5, 6)])
def test_gpu_single_user_is_the_single_user_soft_path(ofdm, detector, dims):
    import torch

    A, N, C, S, b = dims
    F, K, snr = 3, N - 1, 20.0
    nv = noise_var_of(snr, N)
    d = ofdm.synth.make_frames(F, A, N, C, S, b, snr_db=snr, seed=N + 1)
    dev = torch.device("cuda:0")
    with ofdm.LsMrcReceiver(A, N, C, S, b) as r:
        r.set_pilot(d["pilot_asc"])
        r.set_oneshot(0)
        d_rx = torch.from_numpy(d["rx"]).to(dev)
        comb = torch.zeros((F, S - 1, K), dtype=torch.complex64, device=dev)
        llr = torch.zeros((F, S - 1, K, b), dtype=torch.float32, device=dev)
        torch.cuda.synchronize()
        r.demod_frames_device_soft(d_rx, F, comb, llr, noise_var=nv)
        r.sync()
        mu = _run_soft(ofdm, r, d_rx, F, 1, b, detector, nv)
    want = llr.cpu().numpy()
    assert llr_row_err(mu["llr"][:, :, 0], want).max() <= 2e-5


@pytest.mark.gpu
def test_gpu_singular_subcarriers_have_zero_llrs(ofdm):
    A, N, C, S, U, b, F = 8, 256, 32, 6, 2, 4, 2
    K = N - 1
    rng = np.random.default_rng(1)
    h = (rng.standard_normal((F, U, A, K)) + 1j * rng.standard_normal((F, U, A, K))) / np.sqrt(2.0)
    ks = [0, 17, 100, 254]                       # subcarrier index k = bin - 1
    h[:, 1, :, ks] = h[:, 0, :, ks]              # both users on the same channel there
    d = ofdm.synth.make_frames_mu(F, A, N, C, S, b, U, snr_db=None, seed=2, h=h)
    pos = [bin_to_asc_pos(k + 1, N) for k in ks]
    rest = np.setdiff1d(np.arange(K), pos)
    with ofdm.LsMrcReceiver(A, N, C, S, b) as r:
        r.set_pilot(d["pilot_asc"])
        got = _run_soft(ofdm, r, d["rx"], F, U, b, "zf", 1e-3, count=True)
    assert got["n_singular"] == F * len(ks)
    assert (got["llr"][..., pos, :] == 0).all() and (got["sinr"][..., pos] == 0).all()
    assert np.isfinite(got["llr"]).all() and (got["sinr"][..., rest] > 0).all()
    assert (np.abs(got["llr"][..., rest, :2]) > 0).any()


@pytest.mark.gpu
def test_gpu_deterministic_and_interleaved_with_other_calls(ofdm):
    import torch

    A, N, C, S, b = 16, 2048, 144, 8, 4
    K = N - 1
    nv = noise_var_of(20.0, N)
    dev = torch.device("cuda:0")
    su = ofdm.synth.make_frames(3, A, N, C, S, b, snr_db=20.0, seed=5)
    m3 = ofdm.synth.make_frames_mu(3, A, N, C, S, b, 3, snr_db=20.0, seed=6, pilot_asc=su["pilot_asc"])
    m2 = ofdm.synth.make_frames_mu(2, A, N, C, S, b, 2, snr_db=20.0, seed=7, pilot_asc=su["pilot_asc"])
    with ofdm.LsMrcReceiver(A, N, C, S, b) as r:
        r.set_pilot(su["pilot_asc"])

        def single_soft():
            comb = torch.zeros((3, S - 1, K), dtype=torch.complex64, device=dev)
            llr = torch.zeros((3, S - 1, K, b), dtype=torch.float32, device=dev)
            torch.cuda.synchronize()
            r.demod_frames_device_soft(torch.from_numpy(su["rx"]).to(dev), 3, comb, llr, noise_var=nv)
            r.sync()
            return llr.cpu().numpy()

        a3 = _run_soft(ofdm, r, m3["rx"], 3, 3, b, "mmse", nv)
        again = _run_soft(ofdm, r, m3["rx"], 3, 3, b, "mmse", nv)
        s0 = single_soft()
        h2 = _run_hard(ofdm, r, m2["rx"], 2, 2, b, "zf", 0.0)
        a2 = _run_soft(ofdm, r, m2["rx"], 2, 2, b, "zf", nv)         # fewer frames and users right after
        s1 = single_soft()
        b3 = _run_soft(ofdm, r, m3["rx"], 3, 3, b, "mmse", nv)
        h2b = _run_hard(ofdm, r, m2["rx"], 2, 2, b, "zf", 0.0)
    for k in ("combined", "bits", "llr", "sinr"):
        assert a3[k].tobytes() == again[k].tobytes() == b3[k].tobytes(), k
    assert s0.tobytes() == s1.tobytes()
    assert h2["combined"].tobytes() == h2b["combined"].tobytes() == a2["combined"].tobytes()
    ref2 = oracle_mu_soft(m2["rx"], m2["pilot_asc"], C, 2, b, "zf", nv)
    assert llr_row_err(a2["llr"], ref2["llr"]).max() <= max(2e-5, 4e-6 * gram_cond(ref2["hconj"]))


@pytest.mark.gpu
@pytest.mark.parametrize("dims", [(8, 64, 16, 8, 2, 3), (32, 1024, 64, 8, 4, 4), (64, 4096, 288, 7, 4, 2)])
def test_gpu_soft_call_replays_from_a_cuda_graph(ofdm, dims):
    import torch

    A, N, C, S, b, U = dims
    F, K = 2, N - 1
    dev = torch.device("cuda:0")
    user = torch.cuda.Stream(dev)
    g = torch.Generator(device=dev).manual_seed(9)
    inputs = [torch.randn((F, S, A, N + C, 2), device=dev, generator=g) for _ in range(3)]
    rx = torch.empty_like(inputs[0])
    comb = torch.zeros((F, S - U, U, K, 2), device=dev)
    bits = torch.zeros((F, S - U, U, (K * b + 7) // 8), device=dev, dtype=torch.uint8)
    llr = torch.zeros((F, S - U, U, K, b), device=dev)
    sinr = torch.zeros((F, U, K), device=dev)
    outs = (comb, bits, llr, sinr)
    torch.cuda.synchronize(dev)
    with ofdm.LsMrcReceiver(A, N, C, S, b) as r:
        r.set_pilot(ofdm.synth.make_pilot(K, 3))
        r.set_stream(user.cuda_stream)

        def call(nv):
            r.demod_frames_device_mu_soft(rx, F, U, comb, llr, bits, None, sinr, detector="mmse", noise_var=nv)

        with torch.cuda.stream(user):
            rx.copy_(inputs[0])
            call(0.1)                               # first call: scratch allocated outside the capture
        user.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=user):
            call(0.1)
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
                call(0.1)
            user.synchronize()
            assert all(torch.equal(a, o) for a, o in zip(got, outs))
            assert bool(torch.isfinite(llr).all()) and float(llr.abs().max()) > 0
            with torch.cuda.stream(user):                 # noise_var is a kernel argument, not state captured on the host
                call(0.2)
            user.synchronize()
            assert not torch.equal(got[2], llr)
        r.set_stream(None)


@pytest.mark.gpu
def test_gpu_more_frames_than_one_grid_dimension(ofdm):
    """65537 frames: the detector build runs in two grid-y chunks, and its diagonal output must follow the chunk"""
    import torch

    A, N, C, S, U, b, F = 4, 64, 16, 3, 2, 2, 65537
    K = N - 1
    nv = noise_var_of(20.0, N)
    dev = torch.device("cuda:0")
    d = ofdm.synth.make_frames_mu(4, A, N, C, S, b, U, snr_db=20.0, seed=65)
    small = torch.from_numpy(d["rx"]).to(dev)
    big = small[torch.arange(F, device=dev) % 4].contiguous()
    with ofdm.LsMrcReceiver(A, N, C, S, b) as r:
        r.set_pilot(d["pilot_asc"])
        want = _run_soft(ofdm, r, small, 4, U, b, "mmse", nv, want_hconj=False)
        llr = torch.zeros((F, S - U, U, K, b), dtype=torch.float32, device=dev)
        sinr = torch.zeros((F, U, K), dtype=torch.float32, device=dev)
        comb = torch.zeros((F, S - U, U, K), dtype=torch.complex64, device=dev)
        torch.cuda.synchronize()
        assert r.demod_frames_device_mu_soft(big, F, U, comb, llr, None, None, sinr, detector="mmse", noise_var=nv,
                                             count_singular=True) == 0
        for f in (0, 3, 65534, 65535, 65536):
            assert llr[f].cpu().numpy().tobytes() == want["llr"][f % 4].tobytes(), f
            assert sinr[f].cpu().numpy().tobytes() == want["sinr"][f % 4].tobytes(), f
        assert bool((llr[:65536].view(16384, 4, S - U, U, K, b) == torch.from_numpy(want["llr"]).to(dev)).all())
        assert bool((sinr[:65536].view(16384, 4, U, K) == torch.from_numpy(want["sinr"]).to(dev)).all())


@pytest.mark.gpu
def test_gpu_argument_errors(ofdm):
    import torch

    A, N, C, S, b = 4, 64, 16, 6, 2
    K = N - 1
    dev = torch.device("cuda:0")
    rx = torch.zeros((1, S, A, N + C), dtype=torch.complex64, device=dev)
    comb = torch.zeros((1, S - 1, 4, K), dtype=torch.complex64, device=dev)
    llr = torch.zeros((1, S - 1, 4, K, b), dtype=torch.float32, device=dev)
    with ofdm.LsMrcReceiver(A, N, C, S, b) as r:
        with pytest.raises(ofdm.LsmrcError) as e:
            r.demod_frames_device_mu_soft(rx, 1, 1, comb, llr, noise_var=0.1)
        assert e.value.code == -4                                   # LSMRC_ERR_NO_PILOT
        r.set_pilot(ofdm.synth.make_pilot(K, 1))
        with pytest.raises(ofdm.LsmrcError) as e:
            r.demod_frames_device_mu_soft(rx, 1, 2, comb, None, noise_var=0.1)
        assert e.value.code == -1                                   # d_llr NULL
        bad_nv = [0.0, -1.0, float("nan"), float("inf")]
        for U, det, nv in [(0, "zf", 0.1), (17, "zf", 0.1), (5, "zf", 0.1), (6, "zf", 0.1), (2, "bogus", 0.1)] + \
                [(2, det, nv) for det in ("zf", "mmse") for nv in bad_nv]:
            with pytest.raises(ofdm.LsmrcError) as e:
                r.demod_frames_device_mu_soft(rx, 1, U, comb, llr, detector=det, noise_var=nv)
            assert e.value.code == -1, (U, det, nv)                 # LSMRC_ERR_INVALID
        r.demod_frames_device_mu_soft(rx, 0, 2, comb, llr, noise_var=0.1)   # no frames: nothing to do
