"""Multi-user uplink (lsmrc_demod_frames_device_mu): per-user LS channel estimates from time-orthogonal pilots and ZF /
MMSE detection fused with the row FFT.  The CPU oracle is tests/cpp/mu_oracle.c (double-precision detector on top of
the single-user oracle's LS estimate, FFT and demapper), built here into a temporary directory."""
import ctypes
import os
import shutil
import subprocess
import tempfile

import numpy as np
import pytest

from util import assert_bits_match, assert_close, rel_errors

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_LIB = {}


def _mu_lib():
    if "lib" not in _LIB:
        d = tempfile.mkdtemp(prefix="mu_oracle_")
        so = os.path.join(d, "libmu_oracle.so")
        srcs = [os.path.join(ROOT, "tests", "cpp", "mu_oracle.c"), os.path.join(ROOT, "oracle", "cpuls_oracle.c"),
                os.path.join(ROOT, "oracle", "fft_shim.c")]
        subprocess.run([os.environ.get("CC", "gcc"), "-O2", "-fPIC", "-ffp-contract=off", "-pthread", "-shared", "-o", so, *srcs,
                        "-lm"], check=True)
        lib = ctypes.CDLL(so)
        shutil.rmtree(d, ignore_errors=True)  # (the mapping stays valid)
        lib.oracle_demod_frames_mu.restype = ctypes.c_int
        lib.oracle_demod_frames_mu.argtypes = [ctypes.c_void_p, ctypes.c_void_p] + [ctypes.c_int] * 7 + [ctypes.c_double] + \
            [ctypes.c_void_p] * 3
        _LIB["lib"] = lib
    return _LIB["lib"]


def oracle_mu(rx, pilot_asc, cp, n_users, qam_bits, noise_var=0.0):
    """rx [F,S,A,N+C] -> dict(hconj [F,U,A,K], combined [F,S-U,U,K], bits [F,S-U,U,row], n_singular)"""
    rx = np.ascontiguousarray(rx, np.complex64)
    F, S, A, NC = rx.shape
    N = NC - cp
    K, U = N - 1, n_users
    pilot_asc = np.ascontiguousarray(pilot_asc, np.complex64)
    hconj = np.empty((F, U, A, K), np.complex64)
    comb = np.empty((F, S - U, U, K), np.complex64)
    bits = np.zeros((F, S - U, U, (K * qam_bits + 7) // 8), np.uint8)
    bad = _mu_lib().oracle_demod_frames_mu(rx.ctypes.data, pilot_asc.ctypes.data, F, S, A, N, cp, U, qam_bits, float(noise_var),
                                           hconj.ctypes.data, comb.ctypes.data, bits.ctypes.data)
    return {"hconj": hconj, "combined": comb, "bits": bits, "n_singular": bad}


def gram_cond(hconj, noise_var=0.0):
    """largest condition number of G_k = H^H H + lambda I over frames and subcarriers; hconj [F,U,A,K]"""
    h = np.conj(hconj.astype(np.complex128)).transpose(0, 3, 2, 1)  # [F,K,A,U]
    g = np.conj(np.swapaxes(h, -1, -2)) @ h + noise_var * np.eye(h.shape[-1])
    return float(np.linalg.cond(g).max())


def bin_to_asc_pos(bin_idx, N):
    return bin_idx - 1 + N // 2 if bin_idx < N // 2 else bin_idx - N // 2


# ------------------------------------------------------------------------------------------------ CPU
def test_oracle_single_user_is_the_mrc_oracle(ofdm, oracle):
    A, N, C, S, b, F = 8, 64, 16, 6, 4, 2
    d = ofdm.synth.make_frames(F, A, N, C, S, b, snr_db=25.0, seed=11)
    ref = oracle.demod_frames(d["rx"], d["pilot_asc"], b, C)
    got = oracle_mu(d["rx"], d["pilot_asc"], C, 1, b)
    assert got["n_singular"] == 0
    assert np.array_equal(got["hconj"][:, 0], ref["hconj"])
    assert_close(got["combined"][:, :, 0], ref["combined"], "combined", tol=1e-6)
    assert_bits_match(got["bits"][:, :, 0], ref["bits"], ref["combined"], b, "bits", got["combined"][:, :, 0])


@pytest.mark.parametrize("U,A", [(2, 8), (4, 8), (2, 16), (4, 16)])
def test_oracle_recovers_noiseless_constellation(ofdm, U, A):
    N, C, S, b, F = 64, 16, U + 4, 4, 2
    d = ofdm.synth.make_frames_mu(F, A, N, C, S, b, U, snr_db=None, seed=100 + U * A)
    got = oracle_mu(d["rx"], d["pilot_asc"], C, U, b)
    assert got["n_singular"] == 0
    kappa = gram_cond(got["hconj"])
    sent = ofdm.synth.qam_map_indices(d["src_idx"], b)
    mx, _ = rel_errors(got["combined"], sent)
    assert mx <= 1e-5 * kappa, (mx, kappa)
    assert np.array_equal(got["bits"], ofdm.synth.pack_bits_rows(d["src_idx"], b))


def _numpy_detect(rx, pilot_asc, cp, U, lam):
    """independent float64 restatement: FFT, LS, np.linalg.solve per subcarrier; combined [F,S-U,U,K] ascending"""
    from gpu_accel_ofdm_ls_mrc_b200.synth import asc_to_bin, bin_to_asc

    z = np.fft.fft(rx[..., cp:].astype(np.complex128), axis=-1)[..., 1:]        # [F,S,A,K]
    x_bin = asc_to_bin(pilot_asc.astype(np.complex128))
    H = (z[:, :U] / x_bin).transpose(0, 3, 2, 1)                                # [F,K,A,U]
    Hh = np.conj(np.swapaxes(H, -1, -2))                                        # [F,K,U,A]
    G = Hh @ H + lam * np.eye(U)
    W = np.linalg.solve(G, Hh)                                                  # [F,K,U,A]
    y = z[:, U:].transpose(0, 3, 2, 1)                                          # [F,K,A,D]
    x = (W @ y).transpose(0, 3, 2, 1)                                           # [F,D,U,K]
    return bin_to_asc(x), G


@pytest.mark.parametrize("U,A,N", [(4, 16, 64), (8, 32, 256)])
@pytest.mark.parametrize("detector", ["zf", "mmse"])
def test_oracle_matches_numpy_solve(ofdm, U, A, N, detector):
    C, S, b, F = N // 8, U + 3, 4, 2
    lam = 0.05 if detector == "mmse" else 0.0
    d = ofdm.synth.make_frames_mu(F, A, N, C, S, b, U, snr_db=20.0, seed=7 * U + N)
    got = oracle_mu(d["rx"], d["pilot_asc"], C, U, b, lam)
    want, G = _numpy_detect(d["rx"], d["pilot_asc"], C, U, lam)
    kappa = float(np.linalg.cond(G).max())
    mx, l2 = rel_errors(got["combined"], want)
    assert mx <= 1e-5 * max(1.0, kappa) and l2 <= 1e-5, (mx, l2, kappa)


def test_mmse_tends_to_zf(ofdm):
    U, A, N, C, S, b, F = 4, 16, 64, 16, 8, 4, 2
    d = ofdm.synth.make_frames_mu(F, A, N, C, S, b, U, snr_db=15.0, seed=3)
    zf = oracle_mu(d["rx"], d["pilot_asc"], C, U, b)["combined"]
    near = oracle_mu(d["rx"], d["pilot_asc"], C, U, b, 1e-9)["combined"]
    far = oracle_mu(d["rx"], d["pilot_asc"], C, U, b, 0.5)["combined"]
    assert rel_errors(near, zf)[0] <= 1e-6
    assert rel_errors(far, zf)[0] >= 1e-3


@pytest.mark.parametrize("dims", [(2, 4, 64, 16, 5, 4, None, 0), (3, 8, 256, 32, 4, 6, 20.0, 9), (1, 2, 128, 0, 3, 2, 10.0, 4)])
def test_make_frames_mu_single_user_is_make_frames(ofdm, dims):
    F, A, N, C, S, b, snr, seed = dims
    a = ofdm.synth.make_frames(F, A, N, C, S, b, snr_db=snr, seed=seed)
    m = ofdm.synth.make_frames_mu(F, A, N, C, S, b, 1, snr_db=snr, seed=seed)
    assert a["rx"].tobytes() == m["rx"].tobytes()
    assert np.array_equal(a["src_idx"], m["src_idx"][:, :, 0])
    assert np.array_equal(a["h_true"], m["h_true"][:, 0])


def test_abi_exports_the_multi_user_entry_point(ofdm):
    lib = ofdm.load_library()
    assert "lsmrc_demod_frames_device_mu" in ofdm.ABI
    assert hasattr(lib, "lsmrc_demod_frames_device_mu")
    text = open(os.path.join(ROOT, "include", "ofdm_lsmrc.h")).read()
    assert "LSMRC_DETECT_ZF = 0" in text and "LSMRC_DETECT_MMSE = 1" in text


# ------------------------------------------------------------------------------------------------ GPU
def _run_gpu(ofdm, r, rx, F, U, b, detector="zf", noise_var=0.0, want_hconj=True, count=False):
    import torch

    A, N, S = r.cfg.n_ant, r.cfg.fft_size, r.cfg.n_sym
    K = N - 1
    dev = torch.device("cuda:0")
    d_rx = torch.from_numpy(np.ascontiguousarray(rx)).to(dev) if isinstance(rx, np.ndarray) else rx
    nan = float("nan")                      # every output element is written: nothing may be left as filled
    comb = torch.view_as_complex(torch.full((F, S - U, U, K, 2), nan, device=dev))
    bits = torch.full((F, S - U, U, (K * b + 7) // 8), 0xA5, dtype=torch.uint8, device=dev)
    hc = torch.view_as_complex(torch.full((F, U, A, K, 2), nan, device=dev)) if want_hconj else None
    torch.cuda.synchronize()
    bad = r.demod_frames_device_mu(d_rx, F, U, comb, bits, hc, detector=detector, noise_var=noise_var, count_singular=count)
    r.sync()
    return {"combined": comb.cpu().numpy(), "bits": bits.cpu().numpy(), "hconj": hc.cpu().numpy() if want_hconj else None,
            "n_singular": bad}


MU_CASES = [  # (A, N, C, S, U, detector, b)
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
def test_gpu_matches_oracle(ofdm, case):
    A, N, C, S, U, det, b = case
    F = 2 if N >= 2048 else 3
    nv = 0.02 if det == "mmse" else 0.0
    d = ofdm.synth.make_frames_mu(F, A, N, C, S, b, U, snr_db=30.0, seed=A + N + U)
    ref = oracle_mu(d["rx"], d["pilot_asc"], C, U, b, nv)
    assert ref["n_singular"] == 0
    with ofdm.LsMrcReceiver(A, N, C, S, b) as r:
        r.set_pilot(d["pilot_asc"])
        got = _run_gpu(ofdm, r, d["rx"], F, U, b, det, nv, count=True)
    assert got["n_singular"] == 0
    assert_close(got["hconj"], ref["hconj"], "hconj")
    tol = max(1e-5, 4e-6 * gram_cond(ref["hconj"], nv))
    assert_close(got["combined"], ref["combined"], "combined", tol=tol)
    assert_bits_match(got["bits"], ref["bits"], ref["combined"], b, "bits", got["combined"], tol=tol)


@pytest.mark.gpu
@pytest.mark.parametrize("dims", [(4, 64, 16, 16, 2), (16, 1024, 64, 6, 4), (16, 4096, 288, 5, 6)])
def test_gpu_single_user_zf_is_mrc(ofdm, dims):
    import torch

    A, N, C, S, b = dims
    F, K = 3, N - 1
    d = ofdm.synth.make_frames(F, A, N, C, S, b, snr_db=25.0, seed=N)
    dev = torch.device("cuda:0")
    with ofdm.LsMrcReceiver(A, N, C, S, b) as r:
        r.set_pilot(d["pilot_asc"])
        r.set_oneshot(0)
        d_rx = torch.from_numpy(d["rx"]).to(dev)
        comb = torch.zeros((F, S - 1, K), dtype=torch.complex64, device=dev)
        bits = torch.zeros((F, S - 1, (K * b + 7) // 8), dtype=torch.uint8, device=dev)
        hc = torch.zeros((F, A, K), dtype=torch.complex64, device=dev)
        torch.cuda.synchronize()
        r.demod_frames_device(d_rx, F, comb, bits, hc)
        r.sync()
        mu = _run_gpu(ofdm, r, d_rx, F, 1, b)
    assert np.array_equal(mu["hconj"][:, 0], hc.cpu().numpy())
    ref_c = comb.cpu().numpy()
    assert_close(mu["combined"][:, :, 0], ref_c, "combined", tol=1e-6)
    assert_bits_match(mu["bits"][:, :, 0], bits.cpu().numpy(), ref_c, b, "bits", mu["combined"][:, :, 0], tol=1e-6)


@pytest.mark.gpu
def test_gpu_singular_subcarriers(ofdm):
    A, N, C, S, U, b, F = 8, 256, 32, 6, 2, 4, 2
    K = N - 1
    rng = np.random.default_rng(1)
    h = (rng.standard_normal((F, U, A, K)) + 1j * rng.standard_normal((F, U, A, K))) / np.sqrt(2.0)
    ks = [0, 17, 100, 254]                       # subcarrier index k = bin - 1
    h[:, 1, :, ks] = h[:, 0, :, ks]              # both users on the same channel there
    d = ofdm.synth.make_frames_mu(F, A, N, C, S, b, U, snr_db=None, seed=2, h=h)
    ref = oracle_mu(d["rx"], d["pilot_asc"], C, U, b)
    assert ref["n_singular"] == F * len(ks)
    pos = [bin_to_asc_pos(k + 1, N) for k in ks]
    rest = np.setdiff1d(np.arange(K), pos)
    with ofdm.LsMrcReceiver(A, N, C, S, b) as r:
        r.set_pilot(d["pilot_asc"])
        got = _run_gpu(ofdm, r, d["rx"], F, U, b, count=True)
        assert got["n_singular"] == ref["n_singular"]
        assert not got["combined"][..., pos].any()
        assert_close(np.ascontiguousarray(got["combined"][..., rest]), np.ascontiguousarray(ref["combined"][..., rest]), "combined")
        mm = _run_gpu(ofdm, r, d["rx"], F, U, b, "mmse", 0.1, count=True)
    assert mm["n_singular"] == 0
    assert np.isfinite(mm["combined"].view(np.float32)).all()


@pytest.mark.gpu
def test_gpu_30db_four_users_decode_exactly(ofdm):
    A, N, C, S, U, b, F = 64, 1024, 64, 10, 4, 4, 2
    d = ofdm.synth.make_frames_mu(F, A, N, C, S, b, U, snr_db=30.0, seed=30)
    with ofdm.LsMrcReceiver(A, N, C, S, b) as r:
        r.set_pilot(d["pilot_asc"])
        got = _run_gpu(ofdm, r, d["rx"], F, U, b, want_hconj=False)
        again = _run_gpu(ofdm, r, d["rx"], F, U, b, want_hconj=False)
    assert np.array_equal(got["bits"], ofdm.synth.pack_bits_rows(d["src_idx"], b))
    assert got["combined"].tobytes() == again["combined"].tobytes() and got["bits"].tobytes() == again["bits"].tobytes()


@pytest.mark.gpu
def test_gpu_interleaved_single_and_multi_user_calls(ofdm):
    import torch

    A, N, C, S, b = 16, 2048, 144, 8, 4
    K = N - 1
    dev = torch.device("cuda:0")
    su = ofdm.synth.make_frames(3, A, N, C, S, b, snr_db=25.0, seed=5)
    m3 = ofdm.synth.make_frames_mu(3, A, N, C, S, b, 3, snr_db=25.0, seed=6, pilot_asc=su["pilot_asc"])
    m2 = ofdm.synth.make_frames_mu(2, A, N, C, S, b, 2, snr_db=25.0, seed=7, pilot_asc=su["pilot_asc"])
    with ofdm.LsMrcReceiver(A, N, C, S, b) as r:
        r.set_pilot(su["pilot_asc"])

        def single():
            comb = torch.zeros((3, S - 1, K), dtype=torch.complex64, device=dev)
            torch.cuda.synchronize()
            r.demod_frames_device(torch.from_numpy(su["rx"]).to(dev), 3, comb)
            r.sync()
            return comb.cpu().numpy()

        s0 = single()
        a3 = _run_gpu(ofdm, r, m3["rx"], 3, 3, b)
        s1 = single()
        a2 = _run_gpu(ofdm, r, m2["rx"], 2, 2, b)        # fewer frames and users right after
        b3 = _run_gpu(ofdm, r, m3["rx"], 3, 3, b)
        s2 = single()
    assert s0.tobytes() == s1.tobytes() == s2.tobytes()
    assert a3["combined"].tobytes() == b3["combined"].tobytes() and a3["bits"].tobytes() == b3["bits"].tobytes()
    ref2 = oracle_mu(m2["rx"], m2["pilot_asc"], C, 2, b)
    assert_close(a2["combined"], ref2["combined"], "combined", tol=max(1e-5, 4e-6 * gram_cond(ref2["hconj"])))


@pytest.mark.gpu
@pytest.mark.parametrize("dims", [(8, 64, 16, 8, 2, 3), (32, 1024, 64, 8, 4, 4), (64, 4096, 288, 7, 4, 2)])
def test_gpu_multi_user_call_replays_from_a_cuda_graph(ofdm, dims):
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
    hc = torch.zeros((F, U, A, K, 2), device=dev)
    outs = (comb, bits, hc)
    torch.cuda.synchronize(dev)
    with ofdm.LsMrcReceiver(A, N, C, S, b) as r:
        r.set_pilot(ofdm.synth.make_pilot(K, 3))
        r.set_stream(user.cuda_stream)

        def call():
            r.demod_frames_device_mu(rx, F, U, comb, bits, hc, detector="mmse", noise_var=0.1)

        with torch.cuda.stream(user):
            rx.copy_(inputs[0])
            call()                                  # first call: scratch allocated outside the capture
        user.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=user):
            call()
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
                call()
            user.synchronize()
            assert all(torch.equal(a, o) for a, o in zip(got, outs))
            assert bool(torch.isfinite(comb).all()) and float(comb.abs().max()) > 0
        r.set_stream(None)


@pytest.mark.gpu
def test_gpu_argument_errors(ofdm):
    import torch

    A, N, C, S, b = 4, 64, 16, 6, 2
    K = N - 1
    dev = torch.device("cuda:0")
    rx = torch.zeros((1, S, A, N + C), dtype=torch.complex64, device=dev)
    comb = torch.zeros((1, S - 1, 4, K), dtype=torch.complex64, device=dev)
    with ofdm.LsMrcReceiver(A, N, C, S, b) as r:
        with pytest.raises(ofdm.LsmrcError) as e:
            r.demod_frames_device_mu(rx, 1, 1, comb)
        assert e.value.code == -4                                   # LSMRC_ERR_NO_PILOT
        r.set_pilot(ofdm.synth.make_pilot(K, 1))
        for U, det, nv in [(0, "zf", 0.0), (17, "zf", 0.0), (5, "zf", 0.0), (6, "zf", 0.0), (2, "bogus", 0.0), (2, "mmse", 0.0),
                           (2, "mmse", -1.0), (2, "mmse", float("nan")), (2, "mmse", float("inf"))]:
            with pytest.raises(ofdm.LsmrcError) as e:
                r.demod_frames_device_mu(rx, 1, U, comb, detector=det, noise_var=nv)
            assert e.value.code == -1, (U, det, nv)                 # LSMRC_ERR_INVALID
        assert r.lib.lsmrc_demod_frames_device_mu(r.h, rx.data_ptr(), 1, 2, 7, 0.0, None, comb.data_ptr(), None, None) == -1


@pytest.mark.gpu
def test_gpu_two_live_handles_with_different_detector_tiles(ofdm):
    """The shared-memory limit of the detector build is a per-process attribute: two live handles whose calls need
    different large tiles (A = 256 and A = 128 at U = 8), interleaved, must each keep working -- through the multi-user
    call and through lsmrc_zf_create."""
    import torch

    dev = torch.device("cuda:0")
    cases = [(256, 64, 16, 10, 8), (128, 64, 16, 10, 8)]  # (A, N, C, S, U)
    data, handles = [], []
    try:
        for i, (A, N, C, S, U) in enumerate(cases):
            d = ofdm.synth.make_frames_mu(2, A, N, C, S, 2, U, snr_db=30.0, seed=40 + i)
            r = ofdm.LsMrcReceiver(A, N, C, S, 2)
            r.set_pilot(d["pilot_asc"])
            data.append(d)
            handles.append(r)
        first = [_run_gpu(ofdm, r, d["rx"], 2, c[4], 2) for r, d, c in zip(handles, data, cases)]
        for order in ((0, 1), (1, 0)):
            for i in order:
                r, d, c, want = handles[i], data[i], cases[i], first[i]
                got = _run_gpu(ofdm, r, d["rx"], 2, c[4], 2)
                assert got["combined"].tobytes() == want["combined"].tobytes()
                A, U, K = c[0], c[4], c[1] - 1
                x = torch.from_numpy(np.ascontiguousarray(got["hconj"][0])).to(dev)          # [U][A][K]
                hz = torch.zeros((K, U, A), dtype=torch.complex64, device=dev)
                torch.cuda.synchronize()
                assert r.zf_create(x, A, K, U, hz) == 0
                assert bool(torch.isfinite(torch.view_as_real(hz)).all()) and float(hz.abs().max()) > 0
        for want, d, c in zip(first, data, cases):
            ref = oracle_mu(d["rx"], d["pilot_asc"], c[2], c[4], 2)
            assert_close(want["combined"], ref["combined"], "combined", tol=max(1e-5, 4e-6 * gram_cond(ref["hconj"])))
    finally:
        for r in handles:
            r.close()


@pytest.mark.gpu
def test_gpu_more_frames_than_one_grid_dimension(ofdm):
    """65537 frames (more than the 65535 blocks of one grid dimension): every frame is decoded as in a small call."""
    import torch

    A, N, C, S, U, b, F = 4, 64, 16, 3, 2, 2, 65537
    K = N - 1
    dev = torch.device("cuda:0")
    d = ofdm.synth.make_frames_mu(4, A, N, C, S, b, U, snr_db=30.0, seed=65)
    small = torch.from_numpy(d["rx"]).to(dev)
    idx = torch.arange(F, device=dev) % 4
    big = small[idx].contiguous()
    with ofdm.LsMrcReceiver(A, N, C, S, b) as r:
        r.set_pilot(d["pilot_asc"])
        want = _run_gpu(ofdm, r, small, 4, U, b, want_hconj=False)
        comb = torch.zeros((F, S - U, U, K), dtype=torch.complex64, device=dev)
        bits = torch.zeros((F, S - U, U, (K * b + 7) // 8), dtype=torch.uint8, device=dev)
        torch.cuda.synchronize()
        assert r.demod_frames_device_mu(big, F, U, comb, bits, count_singular=True) == 0
        for f in (0, 3, 65532, 65533, 65534, 65535, 65536):
            assert comb[f].cpu().numpy().tobytes() == want["combined"][f % 4].tobytes(), f
            assert bits[f].cpu().numpy().tobytes() == want["bits"][f % 4].tobytes(), f
        whole = comb[:65536].view(16384, 4, S - U, U, K)            # every block of 4 frames equals the small call
        assert bool((whole == torch.from_numpy(want["combined"]).to(dev)).all())
