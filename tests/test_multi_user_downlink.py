"""Multi-user downlink (lsmrc_precode_frames_device): reciprocal ZF / regularised-ZF precoding from the uplink channel
estimate, fused with the inverse row FFT and the cyclic prefix (DESIGN.md 8g).  precode_ref restates the math in
float64 numpy -- np.linalg.solve per subcarrier, np.fft.ifft, CP -- independently of the C oracles; the CPU tests pin it
to the defining property, the single-user closed form, the reference's ZF matrix (oracle.zf_create) and the power rule,
and the GPU tests hold the library to it, then run a loop-back through the project's own receiver."""
import numpy as np
import pytest

from mu_ref64 import precode_ref
from util import rel_errors


def _gram(hconj, reg):
    """G_k = H_k^H H_k + reg I per (frame, subcarrier) from conj(H) [F,U,A,K]: [F,K,U,U]"""
    H = np.conj(hconj.astype(np.complex128)).transpose(0, 3, 2, 1)          # [F,K,A,U]
    return np.conj(np.swapaxes(H, -1, -2)) @ H + reg * np.eye(H.shape[-1])


def gram_cond(hconj, reg=0.0, singular=None):
    c = np.linalg.cond(_gram(hconj, reg))
    if singular is not None:
        c = np.where(singular, 1.0, c)
    return float(c.max())


def _channels(F, U, A, K, seed):
    rng = np.random.default_rng(seed)
    return ((rng.standard_normal((F, U, A, K)) + 1j * rng.standard_normal((F, U, A, K))) / np.sqrt(2.0)).astype(np.complex64)


def _symbols(F, Sd, U, K, b, seed):
    from gpu_accel_ofdm_ls_mrc_b200.synth import qam_map_indices

    idx = np.random.default_rng(seed).integers(0, 1 << b, size=(F, Sd, U, K), dtype=np.uint8)
    return idx, qam_map_indices(idx, b).astype(np.complex64)


def _demap(y, b):
    """nearest constellation point -> index (y [...] complex)"""
    from gpu_accel_ofdm_ls_mrc_b200.synth import qam_map_indices

    pts = qam_map_indices(np.arange(1 << b), b)
    return np.abs(y[..., None] - pts).argmin(axis=-1).astype(np.uint8)


# ------------------------------------------------------------------------------------------------ CPU
@pytest.mark.parametrize("U,A,reg", [(2, 4, 0.0), (4, 16, 0.0), (16, 16, 0.0), (4, 8, 0.3)])
def test_reference_precoder_inverts_the_downlink_channel(ofdm, U, A, reg):
    N, C, F, Sd = 64, 16, 2, 3
    K = N - 1
    hconj = np.conj(_channels(F, U, A, K, 1))
    _, sym = _symbols(F, Sd, U, K, 4, 2)
    ref = precode_ref(hconj, sym, reg, N, C)
    assert not ref["singular"].any()
    H = np.conj(hconj.astype(np.complex128)).transpose(0, 3, 2, 1)          # [F,K,A,U]
    HtP = np.swapaxes(H, -1, -2) @ ref["P"]                                  # downlink channel times precoder
    cond = np.linalg.cond(_gram(hconj, reg))
    if reg == 0.0:
        assert (np.abs(HtP - np.eye(U)).max(axis=(-1, -2)) <= 1e-12 * cond).all()
    else:                                                                    # regularised: H^T P = I - reg conj(inv(G))
        want = np.eye(U) - reg * np.conj(np.linalg.inv(_gram(hconj, reg)))
        assert np.abs(HtP - want).max() <= 1e-12 * cond.max()
    # the transmitted rows: the receiver's unnormalised FFT of a row (CP dropped) gives back g z; CP = the row's tail
    tx = ref["tx"]
    assert np.array_equal(tx[..., :C], tx[..., N:N + C])
    back = np.fft.fft(tx[..., C:], axis=-1)
    assert np.abs(back - ref["gain"][:, None, None, None] * ref["z"]).max() <= 1e-12 * np.abs(back).max()


def test_reference_single_user_closed_form(ofdm):
    N, C, F, Sd, A = 128, 16, 2, 2, 8
    K = N - 1
    hconj = np.conj(_channels(F, 1, A, K, 3))
    _, sym = _symbols(F, Sd, 1, K, 2, 4)
    ref = precode_ref(hconj, sym, 0.0, N, C)
    h = np.conj(hconj[:, 0].astype(np.complex128)).transpose(0, 2, 1)      # [F,K,A]
    want = np.conj(h) / (np.abs(h) ** 2).sum(axis=-1, keepdims=True)
    assert np.abs(ref["P"][..., 0] - want).max() <= 1e-13 * np.abs(want).max()


@pytest.mark.parametrize("U,A,K", [(1, 1, 7), (2, 4, 63), (4, 16, 255), (16, 16, 31)])
def test_reference_precoder_is_the_reference_zf_matrix(ofdm, oracle, U, A, K):
    """createZeroForcingMatrix on X = conj(H) [U][A][K] is the precoder: P_k[a][u] = conj(Hzf[k][u][a])"""
    N = K + 1
    hconj = np.conj(_channels(1, U, A, K, 5))
    _, sym = _symbols(1, 1, U, K, 2, 6)
    P = precode_ref(hconj, sym, 0.0, N, 0)["P"][0]                           # [K,A,U]
    Hzf, bad = oracle.zf_create(hconj[0])                                     # X = conj(H), [U][A][K]
    assert bad == 0
    want = np.conj(Hzf.astype(np.complex128)).transpose(0, 2, 1)             # [K,A,U]
    cond = gram_cond(hconj)
    assert np.abs(P - want).max() <= 2e-7 * cond * np.abs(P).max(), (np.abs(P - want).max(), cond)


def test_reference_power_rule(ofdm):
    U, A, N, C, F, Sd = 3, 8, 256, 32, 3, 2
    K = N - 1
    h = _channels(F, U, A, K, 7)
    ks = [0, 40, 200]
    h[1, 2][:, ks] = h[1, 0][:, ks]                                          # singular subcarriers in frame 1 only
    hconj = np.conj(h)
    _, sym = _symbols(F, Sd, U, K, 4, 8)
    for reg in (0.0, 0.05):
        ref = precode_ref(hconj, sym, reg, N, C)
        assert ref["singular"].sum() == (len(ks) if reg == 0.0 else 0)
        total = (np.abs(ref["gain"][:, None, None, None] * ref["P"]) ** 2).sum(axis=(1, 2, 3))
        assert np.allclose(total, U * K, rtol=1e-12, atol=0)
    # unit-energy symbols: mean transmit energy per used subcarrier is U on average over a long frame
    _, many = _symbols(1, 400, U, K, 4, 9)
    ref = precode_ref(hconj[:1], many, 0.0, N, C)
    energy = (np.abs(np.fft.fft(ref["tx"][..., C:], axis=-1)[..., 1:]) ** 2).sum(axis=(2, 3)).mean() / K
    assert abs(energy - U) <= 0.05 * U


# ------------------------------------------------------------------------------------------------ GPU
GUARD = 4096  # NaN elements after d_tx and d_gain that no call may touch


def _run_gpu(r, hconj, sym, reg, count=True, want_gain=True):
    import torch

    F, U, A, K = hconj.shape
    Sd = sym.shape[1]
    N, C = r.cfg.fft_size, r.cfg.cp_len
    dev = torch.device("cuda:0")
    d_h = torch.from_numpy(np.ascontiguousarray(hconj, np.complex64)).to(dev) if isinstance(hconj, np.ndarray) else hconj
    d_s = torch.from_numpy(np.ascontiguousarray(sym, np.complex64)).to(dev) if isinstance(sym, np.ndarray) else sym
    n_tx = F * Sd * A * (N + C) * 2
    tx_buf = torch.full((n_tx + GUARD,), float("nan"), device=dev)
    gain_buf = torch.full((F + GUARD,), float("nan"), device=dev)
    tx, gain = tx_buf[:n_tx], (gain_buf[:F] if want_gain else None)
    torch.cuda.synchronize()
    bad = r.precode_frames_device(d_h, F, U, d_s, Sd, tx, gain, reg=reg, count_singular=count)
    r.sync()
    assert bool(torch.isnan(tx_buf[n_tx:]).all()) and bool(torch.isnan(gain_buf[F:]).all()), "a write past d_tx or d_gain"
    return {"tx": torch.view_as_complex(tx.view(F, Sd, A, N + C, 2)).cpu().numpy(), "gain": gain.cpu().numpy() if want_gain else None,
            "n_singular": bad}


DL_CASES = [  # (A, N, C, U, Sd, reg)
    (4, 64, 16, 1, 3, 0.0),
    (8, 64, 16, 2, 2, 0.05),
    (16, 64, 16, 16, 2, 0.0),
    (8, 128, 16, 4, 3, 0.1),
    (16, 128, 0, 2, 2, 0.0),
    (16, 256, 32, 4, 2, 0.0),
    (32, 512, 32, 2, 2, 0.05),
    (64, 1024, 64, 4, 2, 0.0),
    (16, 1024, 64, 16, 1, 0.1),
    (16, 2048, 144, 2, 2, 0.0),
    (32, 2048, 144, 4, 2, 0.1),
    (32, 4096, 288, 2, 2, 0.0),
    (64, 4096, 288, 4, 2, 0.05),
    # odd user counts on every plan: the precoder rows of frame f start at f * U (not at the uplink's padded group count)
    (8, 64, 16, 3, 2, 0.0),
    (24, 64, 16, 9, 2, 0.05),
    (16, 128, 16, 5, 2, 0.0),
    (16, 256, 32, 7, 2, 0.1),
    (32, 256, 32, 15, 1, 0.0),
    (16, 512, 32, 5, 2, 0.05),
    (8, 1024, 64, 3, 2, 0.0),
    (32, 1024, 64, 15, 2, 0.1),
    (16, 2048, 144, 7, 2, 0.0),
    (20, 4096, 288, 9, 2, 0.05),
    (16, 4096, 288, 5, 1, 0.0),
]


@pytest.mark.gpu
@pytest.mark.parametrize("case", DL_CASES, ids=lambda c: "A{}_N{}_C{}_U{}_Sd{}_reg{}".format(*c))
def test_gpu_matches_reference(ofdm, case):
    A, N, C, U, Sd, reg = case
    F, K = 3, N - 1
    hconj = np.conj(_channels(F, U, A, K, A + N + U))
    _, sym = _symbols(F, Sd, U, K, 4, N + U)
    ref = precode_ref(hconj, sym, reg, N, C)
    assert not ref["singular"].any()
    with ofdm.LsMrcReceiver(A, N, C, 2, 2) as r:
        got = _run_gpu(r, hconj, sym, reg)
        again = _run_gpu(r, hconj, sym, reg, count=False, want_gain=False)
    assert got["n_singular"] == 0
    tx = got["tx"]
    assert np.isfinite(tx.view(np.float32)).all(), "every sample is written"
    assert tx[..., :C].tobytes() == tx[..., N:N + C].tobytes(), "the cyclic prefix is the row's tail, bit for bit"
    assert again["tx"].tobytes() == tx.tobytes(), "d_gain = NULL gives the same samples"
    tol = max(1e-5, 4e-6 * gram_cond(hconj, reg))
    for f in range(F):                      # each frame against its own scale
        mx, l2 = rel_errors(tx[f], ref["tx"][f])
        assert mx <= tol and l2 <= tol, (f, mx, l2, tol)
    assert np.abs(got["gain"] - ref["gain"]).max() <= tol * ref["gain"].max(), (got["gain"], ref["gain"])


def _fft_rows(r, tx):
    """the library's own CP strip and forward FFT of tx [F,Sd,A,N+C] (device tensor) -> [F,Sd,A,N] numpy"""
    import torch

    F, Sd, A, NC = tx.shape
    N = r.cfg.fft_size
    rows = F * Sd * A
    out = torch.empty((F, Sd, A, N), dtype=torch.complex64, device=tx.device)
    torch.cuda.synchronize()
    r.stage("drop_prefix", out, tx, rows)
    r.stage("fft", out, rows)
    r.sync()
    return out.cpu().numpy().astype(np.complex128)


@pytest.mark.gpu
@pytest.mark.parametrize("dims", [(32, 1024, 64, 4, 4), (16, 2048, 144, 2, 4), (32, 4096, 288, 4, 2)])
def test_gpu_loop_back_through_the_receiver(ofdm, dims):
    """Uplink pilots -> lsmrc_demod_frames_device_mu -> exported conj(H) -> precode -> the library's FFT of tx -> each
    user's true downlink channel H_k^T -> / g_f -> demap: every user recovers its bits.  Noiseless uplink: the
    per-user error is at the fp32 rounding level."""
    import torch

    A, N, C, U, b = dims
    F, Sd, K = 2, 3, N - 1
    dev = torch.device("cuda:0")
    idx, sym = _symbols(F, Sd, U, K, b, 31 + N)
    for snr in (30.0, None):
        up = ofdm.synth.make_frames_mu(F, A, N, C, U + 1, b, U, snr_db=snr, seed=17 + N)
        h = up["h_true"]                                                     # [F,U,A,K] bin order
        with ofdm.LsMrcReceiver(A, N, C, U + 1, b) as r:
            r.set_pilot(up["pilot_asc"])
            d_rx = torch.from_numpy(up["rx"]).to(dev)
            hc = torch.zeros((F, U, A, K), dtype=torch.complex64, device=dev)
            comb = torch.zeros((F, 1, U, K), dtype=torch.complex64, device=dev)
            d_sym = torch.from_numpy(sym).to(dev)
            tx = torch.zeros((F, Sd, A, N + C), dtype=torch.complex64, device=dev)
            gain = torch.zeros((F,), dtype=torch.float32, device=dev)
            torch.cuda.synchronize()
            r.demod_frames_device_mu(d_rx, F, U, comb, None, hc)
            assert r.precode_frames_device(hc, F, U, d_sym, Sd, tx, gain, count_singular=True) == 0
            y = _fft_rows(r, tx)                                             # [F,Sd,A,N]
            g = gain.cpu().numpy().astype(np.float64)
        rx_user = np.einsum("fuak,fdak->fduk", h, y[..., 1:]) / g[:, None, None, None]     # bin order
        from gpu_accel_ofdm_ls_mrc_b200.synth import bin_to_asc

        est = bin_to_asc(rx_user)
        if snr is not None:
            assert np.array_equal(_demap(est, b), idx), "bit errors at 30 dB"
        else:
            err = np.abs(est - sym).max() / np.abs(sym).max()
            kappa = gram_cond(np.conj(h))
            assert err <= 1e-5 * kappa, (err, kappa)


@pytest.mark.gpu
@pytest.mark.parametrize("N,C", [(256, 32), (4096, 288)])
def test_gpu_singular_subcarriers(ofdm, N, C):
    A, U, F, Sd = 8, 2, 2, 2
    K = N - 1
    h = _channels(F, U, A, K, 13)
    ks = [0, 17, 100, K - 1]                                                  # subcarrier index k = bin - 1
    h[:, 1][:, :, ks] = h[:, 0][:, :, ks]                                     # both users on the same channel there
    hconj = np.conj(h)
    _, sym = _symbols(F, Sd, U, K, 4, 14)
    ref = precode_ref(hconj, sym, 0.0, N, C)
    assert ref["singular"].sum() == F * len(ks)
    with ofdm.LsMrcReceiver(A, N, C, 2, 2) as r:
        got = _run_gpu(r, hconj, sym, 0.0)
        rg = _run_gpu(r, hconj, sym, 0.2)
    assert got["n_singular"] == F * len(ks) and rg["n_singular"] == 0
    spec = np.fft.fft(got["tx"][..., C:].astype(np.complex128), axis=-1)
    bins = [k + 1 for k in ks]
    assert np.abs(spec[..., bins]).max() <= 1e-5 * np.abs(spec).max()
    tol = max(1e-5, 4e-6 * gram_cond(hconj, 0.0, ref["singular"]))
    assert rel_errors(got["tx"], ref["tx"])[0] <= tol
    assert np.abs(got["gain"] - ref["gain"]).max() <= tol * ref["gain"].max()
    assert rel_errors(rg["tx"], precode_ref(hconj, sym, 0.2, N, C)["tx"])[0] <= max(1e-5, 4e-6 * gram_cond(hconj, 0.2))


@pytest.mark.gpu
def test_gpu_all_singular_frame_transmits_nothing(ofdm):
    A, N, C, U, F, Sd = 4, 64, 16, 2, 2, 1
    K = N - 1
    h = _channels(F, U, A, K, 21)
    h[1, 1] = h[1, 0]                                                         # frame 1: every subcarrier singular
    _, sym = _symbols(F, Sd, U, K, 2, 22)
    with ofdm.LsMrcReceiver(A, N, C, 2, 2) as r:
        got = _run_gpu(r, np.conj(h), sym, 0.0)
    assert got["n_singular"] == K
    assert got["gain"][1] == 0.0 and got["gain"][0] > 0
    assert not got["tx"][1].any() and got["tx"][0].any()


@pytest.mark.gpu
def test_gpu_repeatable_and_interleaved_with_the_uplink(ofdm):
    import torch

    A, N, C, S, b = 16, 2048, 144, 6, 4
    K = N - 1
    dev = torch.device("cuda:0")
    m3 = ofdm.synth.make_frames_mu(3, A, N, C, S, b, 3, snr_db=25.0, seed=5)
    with ofdm.LsMrcReceiver(A, N, C, S, b) as r:
        r.set_pilot(m3["pilot_asc"])

        def uplink():
            comb = torch.zeros((3, S - 3, 3, K), dtype=torch.complex64, device=dev)
            hc = torch.zeros((3, 3, A, K), dtype=torch.complex64, device=dev)
            torch.cuda.synchronize()
            r.demod_frames_device_mu(torch.from_numpy(m3["rx"]).to(dev), 3, 3, comb, None, hc)
            r.sync()
            return comb.cpu().numpy(), hc.cpu().numpy()

        u0, hc = uplink()
        _, sym3 = _symbols(3, 4, 3, K, 4, 1)
        _, sym2 = _symbols(2, 2, 2, K, 4, 2)
        a = _run_gpu(r, hc, sym3, 0.0)
        u1, _ = uplink()
        c = _run_gpu(r, np.ascontiguousarray(hc[:2, :2]), sym2, 0.1)         # fewer frames, users and symbols right after
        b2 = _run_gpu(r, hc, sym3, 0.0)
        u2, _ = uplink()
    assert u0.tobytes() == u1.tobytes() == u2.tobytes()
    assert a["tx"].tobytes() == b2["tx"].tobytes() and a["gain"].tobytes() == b2["gain"].tobytes()
    ref = precode_ref(hc[:2, :2], sym2, 0.1, N, C)
    assert rel_errors(c["tx"], ref["tx"])[0] <= max(1e-5, 4e-6 * gram_cond(hc[:2, :2], 0.1))


@pytest.mark.gpu
@pytest.mark.parametrize("dims", [(8, 64, 16, 2, 3), (32, 1024, 64, 4, 2), (64, 4096, 288, 4, 2)])
def test_gpu_precode_call_replays_from_a_cuda_graph(ofdm, dims):
    import torch

    A, N, C, U, Sd = dims
    F, K = 2, N - 1
    dev = torch.device("cuda:0")
    user = torch.cuda.Stream(dev)
    g = torch.Generator(device=dev).manual_seed(9)
    inputs = [(torch.randn((F, U, A, K, 2), device=dev, generator=g), torch.randn((F, Sd, U, K, 2), device=dev, generator=g))
              for _ in range(3)]
    hc = torch.empty_like(inputs[0][0])
    sym = torch.empty_like(inputs[0][1])
    tx = torch.zeros((F, Sd, A, N + C, 2), device=dev)
    gain = torch.zeros((F,), device=dev)
    outs = (tx, gain)
    torch.cuda.synchronize(dev)
    with ofdm.LsMrcReceiver(A, N, C, 2, 2) as r:
        r.set_stream(user.cuda_stream)

        def call():
            r.precode_frames_device(hc, F, U, sym, Sd, tx, gain, reg=0.01)

        with torch.cuda.stream(user):
            hc.copy_(inputs[0][0])
            sym.copy_(inputs[0][1])
            call()                                  # first call: scratch allocated outside the capture
        user.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=user):
            call()
        for x, s in inputs:
            with torch.cuda.stream(user):
                hc.copy_(x)
                sym.copy_(s)
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
            assert bool(torch.isfinite(tx).all()) and float(tx.abs().max()) > 0
        r.set_stream(None)


@pytest.mark.gpu
def test_gpu_more_frames_than_one_grid_dimension(ofdm):
    """65537 frames (more than the 65535 blocks of one grid dimension of the precoder build): every frame is precoded
    as in a small call."""
    import torch

    A, N, C, U, Sd, F = 4, 64, 16, 2, 1, 65537
    K = N - 1
    dev = torch.device("cuda:0")
    hconj = np.conj(_channels(4, U, A, K, 65))
    _, sym = _symbols(4, Sd, U, K, 2, 66)
    with ofdm.LsMrcReceiver(A, N, C, 2, 2) as r:
        want = _run_gpu(r, hconj, sym, 0.0)
        idx = torch.arange(F, device=dev) % 4
        big_h = torch.from_numpy(hconj).to(dev)[idx].contiguous()
        big_s = torch.from_numpy(sym).to(dev)[idx].contiguous()
        tx = torch.zeros((F, Sd, A, N + C), dtype=torch.complex64, device=dev)
        gain = torch.zeros((F,), dtype=torch.float32, device=dev)
        torch.cuda.synchronize()
        assert r.precode_frames_device(big_h, F, U, big_s, Sd, tx, gain, count_singular=True) == 0
        for f in (0, 3, 65532, 65533, 65534, 65535, 65536):
            assert tx[f].cpu().numpy().tobytes() == want["tx"][f % 4].tobytes(), f
            assert gain[f].item() == want["gain"][f % 4], f
        whole = tx[:65536].view(16384, 4, Sd, A, N + C)
        assert bool((whole == torch.from_numpy(want["tx"].astype(np.complex64)).to(dev)).all())


@pytest.mark.gpu
def test_gpu_argument_errors(ofdm):
    import torch

    A, N, C = 4, 64, 16
    K = N - 1
    dev = torch.device("cuda:0")
    hc = torch.ones((1, 4, A, K), dtype=torch.complex64, device=dev)
    sym = torch.ones((1, 2, 4, K), dtype=torch.complex64, device=dev)
    tx = torch.zeros((1, 2, A, N + C), dtype=torch.complex64, device=dev)
    with ofdm.LsMrcReceiver(A, N, C, 2, 2) as r:
        before = r.launch_count()
        for U, Sd, reg in [(0, 1, 0.0), (17, 1, 0.0), (5, 1, 0.0), (2, 0, 0.0), (2, 1, -1.0), (2, 1, float("nan")),
                           (2, 1, float("inf")), (2, 1, -float("inf"))]:
            with pytest.raises(ofdm.LsmrcError) as e:
                r.precode_frames_device(hc, 1, U, sym, Sd, tx, reg=reg)
            assert e.value.code == -1, (U, Sd, reg)                          # LSMRC_ERR_INVALID
        p = r.lib.lsmrc_precode_frames_device
        assert p(r.h, None, 1, 2, 0.0, sym.data_ptr(), 1, tx.data_ptr(), None, None) == -1
        assert p(r.h, hc.data_ptr(), 1, 2, 0.0, None, 1, tx.data_ptr(), None, None) == -1
        assert p(r.h, hc.data_ptr(), 1, 2, 0.0, sym.data_ptr(), 1, None, None, None) == -1
        assert r.launch_count() == before, "nothing is launched for a rejected call"
