"""Multi-user uplink with comb pilots (lsmrc_set_mu_pilots(h, LSMRC_MU_PILOTS_COMB), DESIGN.md 8h): all users send
their pilot in symbol 0, user u on the ascending-frequency indices i = u mod U, and the receiver interpolates each
user's channel across its own comb.  comb_ref (mu_ref64.py) restates the whole chain in float64 numpy -- CP strip, np.fft.fft, LS on
symbol 0, the interpolation rule, np.linalg.solve per subcarrier, hard decisions -- independently of the library and of
the C oracles.  The CPU tests pin the rule and the generator and measure the interpolation error of the multipath
settings the GPU tests decode; the GPU tests hold the library to comb_ref on every plan."""
import numpy as np
import pytest

from mu_ref64 import _synth, comb_ref, demap, interp_comb, phi, soft_ref
from util import assert_bits_match, assert_close


def noise_var_of(snr_db, N):
    """noise variance per antenna and subcarrier after the FFT of synth.make_frames_mu's AWGN at snr_db"""
    return (N - 1) / N * 10.0 ** (-snr_db / 10.0)


def llr_row_err(got, ref):
    """largest |got - ref| of each LLR row (last two axes [K, b]) over that row's max |ref|"""
    d = np.abs(got.astype(np.float64) - ref).max(axis=(-1, -2))
    return d / np.maximum(np.abs(ref).max(axis=(-1, -2)), 1e-30)


def comb_frames(F, A, N, C, S, b, U, snr_db, seed, n_taps=4, h=None):
    synth = _synth()
    if h is None:
        h = synth.multipath_channel(F, U, A, N, n_taps, seed=seed + 1000)
    return synth.make_frames_mu(F, A, N, C, S, b, U, snr_db=snr_db, seed=seed, h=h, pilots="comb")


# ------------------------------------------------------------------------------------------------ CPU
@pytest.mark.parametrize("U,N", [(1, 64), (3, 64), (4, 256), (16, 64), (16, 1024)])
def test_rule_is_exact_on_own_pilots_and_constants(U, N):
    K = N - 1
    rng = np.random.default_rng(U + N)
    ls = rng.standard_normal((2, K)) + 1j * rng.standard_normal((2, K))
    out = interp_comb(ls, U, N)
    for u in range(U):
        assert np.array_equal(out[:, u, u::U], ls[:, u::U])                   # own pilots: copied
    if U == 1:
        assert np.array_equal(out[:, 0], ls)
    const = np.broadcast_to(np.array([0.3 - 1.1j, 2.0 + 0.5j])[:, None], (2, K))
    assert np.array_equal(interp_comb(const, U, N), np.broadcast_to(const[:, None], (2, U, K)))


@pytest.mark.parametrize("U,N", [(2, 64), (5, 128), (16, 64), (8, 4096)])
def test_rule_is_exact_for_channels_linear_in_phi_and_holds_the_edges(U, N):
    K = N - 1
    ph = phi(np.arange(K), N).astype(np.float64)
    lin = (0.25 - 0.5j) + (0.01 + 0.02j) * ph
    out = interp_comb(lin, U, N)
    for u in range(U):
        own = np.arange(u, K, U)
        inner = (np.arange(K) >= own[0]) & (np.arange(K) <= own[-1])
        assert np.abs(out[u, inner] - lin[inner]).max() <= 1e-12               # linear between pilots, DC step included
        assert np.array_equal(out[u, : own[0]], np.full(own[0], lin[own[0]]))  # held below the first pilot
        assert np.array_equal(out[u, own[-1]:], np.full(K - own[-1], lin[own[-1]]))   # and above the last


def test_rule_steps_over_dc():
    """Across DC phi jumps by 2: a user whose pilots sit at i = N/2 - 1 (phi = -1) and N/2 + 1 (phi = +2) gets
    w = 2/3 at i = N/2 (phi = +1), not 1/2."""
    N, U = 64, 2
    K = N - 1
    u = (N // 2 - 1) % U
    ls = np.zeros(K, np.complex128)
    ls[N // 2 - 1], ls[N // 2 + 1] = 0.0, 3.0
    assert phi(N // 2 - 1, N) == -1 and phi(N // 2, N) == 1 and phi(N // 2 + 1, N) == 2
    assert interp_comb(ls, U, N)[u, N // 2] == 2.0


@pytest.mark.parametrize("U,A,N", [(1, 2, 64), (4, 3, 64), (16, 2, 256)])
def test_noiseless_comb_frames_give_the_channel_on_each_comb(ofdm, U, A, N):
    synth = ofdm.synth
    F, C, S, b = 2, 16, 3, 4
    K = N - 1
    d = synth.make_frames_mu(F, A, N, C, S, b, U, snr_db=None, seed=U, pilots="comb")
    assert d["src_idx"].shape == (F, S - 1, U, K)
    z = np.fft.fft(d["rx"][..., C:].astype(np.complex128), axis=-1)[..., 1:]
    ratio = synth.bin_to_asc(z[:, 0] / synth.asc_to_bin(d["pilot_asc"].astype(np.complex128)))    # [F,A,K] ascending
    h_asc = synth.bin_to_asc(d["h_true"])                                                           # [F,U,A,K]
    for u in range(U):
        assert np.abs(ratio[..., u::U] - h_asc[:, u, :, u::U]).max() <= 1e-5
    if U == 1:                                           # every subcarrier a pilot: the time-orthogonal frame at U = 1
        t = synth.make_frames_mu(F, A, N, C, S, b, 1, snr_db=None, seed=U)
        assert t["rx"].tobytes() == d["rx"].tobytes()
        ref = comb_ref(d["rx"], d["pilot_asc"], C, U, 0.0, b)
        assert np.abs(ref["combined"] - synth.qam_map_indices(d["src_idx"], b)).max() <= 1e-5


def test_time_default_is_unchanged(ofdm):
    a = ofdm.synth.make_frames_mu(2, 4, 64, 16, 6, 4, 3, snr_db=20.0, seed=5)
    b = ofdm.synth.make_frames_mu(2, 4, 64, 16, 6, 4, 3, snr_db=20.0, seed=5, pilots="time")
    assert a["rx"].tobytes() == b["rx"].tobytes() and np.array_equal(a["src_idx"], b["src_idx"])
    with pytest.raises(ValueError):
        ofdm.synth.make_frames_mu(1, 4, 64, 16, 6, 4, 3, pilots="dft")


def test_multipath_channel_is_a_tapped_delay_line(ofdm):
    F, U, A, N, L = 3, 2, 4, 256, 5
    h = ofdm.synth.multipath_channel(F, U, A, N, L, seed=3)
    assert h.shape == (F, U, A, N - 1)
    full = np.zeros((F, U, A, N), np.complex128)
    full[..., 1:] = h
    full[..., 0] = h.mean(-1) * 0          # bin 0 unknown: reconstruct the taps from bins 1..N-1 by least squares
    k = np.arange(1, N)
    E = np.exp(-2j * np.pi * np.outer(k, np.arange(L)) / N)                   # [K,L]
    taps = np.linalg.lstsq(E, h.reshape(-1, N - 1).T, rcond=None)[0]          # [L, F*U*A]
    assert np.abs(E @ taps - h.reshape(-1, N - 1).T).max() <= 1e-12           # exactly L taps at delays 0..L-1
    big = ofdm.synth.multipath_channel(200, 1, 8, 64, 4, seed=4)
    assert abs((np.abs(big) ** 2).mean() - 1.0) <= 0.05                      # normalised power


# The GPU decoding tests' settings: (A, N, C, S, U, b, snr, seed, taps).  For each, comb_ref (float64) must decode every
# bit with a margin well above fp32 rounding, and its interpolation error must stay within the DESIGN 8h bounds.
DECODE_CASES = [(64, 1024, 64, 6, 8, 4, 30.0, 81, 4), (64, 1024, 64, 6, 16, 4, 30.0, 82, 4)]
LOOPBACK_CASE = (32, 1024, 64, 2, 4, 4, 30.0, 83, 4)   # (A, N, C, S, U, b, snr, seed, taps)


def interp_bounds(U, N, L):
    """DESIGN 8h, per unit of sum_l |g_l| (the taps of a channel with delays < L): linear interpolation between pilots
    at most (2 pi (L-1) D / N)^2 / 8 with D = U + 1 (the spacing across DC; U elsewhere), holding beyond the outermost
    pilots at most 2 pi (L-1) (U-1) / N (a first-order error over at most U-1 subcarriers)"""
    return (2 * np.pi * (L - 1) * (U + 1) / N) ** 2 / 8, 2 * np.pi * (L - 1) * (U - 1) / N


@pytest.mark.parametrize("case", DECODE_CASES + [LOOPBACK_CASE], ids=lambda c: "A{}_N{}_U{}".format(c[0], c[1], c[4]))
def test_reference_interpolation_error_of_the_gpu_settings(ofdm, case):
    from util import symbol_margins

    A, N, C, S, U, b, snr, seed, L = case
    F, K = 2, N - 1
    synth = ofdm.synth
    d = comb_frames(F, A, N, C, S, b, U, None, seed, n_taps=L)
    ref = comb_ref(d["rx"], d["pilot_asc"], C, U, 0.0, b)                     # noiseless: interpolation error only
    h = d["h_true"]
    E = np.exp(-2j * np.pi * np.outer(np.arange(1, N), np.arange(L)) / N)    # [K,L]
    taps = np.linalg.lstsq(E, h.reshape(-1, K).T, rcond=None)[0]             # [L, F*U*A]
    gsum = np.abs(taps).sum(0).reshape(F, U, A, 1)
    err = synth.bin_to_asc(np.abs(np.conj(ref["hconj"]) - h)) / gsum          # [F,U,A,K] ascending
    b_in, b_edge = interp_bounds(U, N, L)
    i = np.arange(K)
    for u in range(U):
        last = u + (K - 1 - u) // U * U
        inner = (i >= u) & (i <= last)
        assert err[:, u][..., inner].max() <= b_in + 1e-6, (u, err[:, u][..., inner].max(), b_in)
        if (~inner).any():
            assert err[:, u][..., ~inner].max() <= b_edge + 1e-6, (u, err[:, u][..., ~inner].max(), b_edge)
    noisy = comb_frames(F, A, N, C, S, b, U, snr, seed, n_taps=L)
    r = comb_ref(noisy["rx"], noisy["pilot_asc"], C, U, 0.0, b)
    assert r["n_singular"] == 0
    if case == LOOPBACK_CASE:                        # ZF precoder from the estimate, applied to the true channel
        H = np.conj(r["hconj"]).transpose(0, 3, 2, 1)                          # [F,K,A,U] estimate
        Ht = noisy["h_true"].transpose(0, 3, 2, 1)                             # [F,K,A,U] truth
        P = np.conj(H) @ np.linalg.inv(np.swapaxes(H, -1, -2) @ np.conj(H))   # [F,K,A,U]
        eff = np.swapaxes(Ht, -1, -2) @ P                                      # [F,K,U,U], I without estimation error
        rng = np.random.default_rng(seed)
        idx = rng.integers(0, 1 << b, size=(F, K, U, 3))
        s = ofdm.synth.qam_map_indices(idx, b)
        y = eff @ s
        assert np.array_equal(demap(y, b), idx)
        assert float(symbol_margins(y, b).min()) >= 0.02
        return
    assert np.array_equal(r["bits"], ofdm.synth.pack_bits_rows(noisy["src_idx"], b))
    assert float(symbol_margins(r["combined"], b).min()) >= 0.02               # fp32 moves a symbol by ~1e-5


def test_abi_exports_the_pilot_layout_setter(ofdm):
    import os

    lib = ofdm.load_library()
    assert "lsmrc_set_mu_pilots" in ofdm.ABI and hasattr(lib, "lsmrc_set_mu_pilots")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    text = open(os.path.join(root, "include", "ofdm_lsmrc.h")).read()
    assert "LSMRC_MU_PILOTS_TIME = 0" in text and "LSMRC_MU_PILOTS_COMB = 1" in text


# ------------------------------------------------------------------------------------------------ GPU
def _dev():
    import torch

    return torch.device("cuda:0")


def _to_dev(x):
    import torch

    return torch.from_numpy(np.ascontiguousarray(x)).to(_dev()) if isinstance(x, np.ndarray) else x


def _run(r, rx, F, U, b, detector="zf", noise_var=0.0, soft=False, count=False, P=1):
    """one multi-user call on the handle's current layout (P pilot symbols) -> dict of host arrays"""
    import torch

    A, N, S = r.cfg.n_ant, r.cfg.fft_size, r.cfg.n_sym
    K, D = N - 1, S - P
    dev = _dev()
    nan = float("nan")                      # every output element is written: nothing may be left as filled
    comb = torch.view_as_complex(torch.full((F, D, U, K, 2), nan, device=dev))
    bits = torch.full((F, D, U, (K * b + 7) // 8), 0xA5, dtype=torch.uint8, device=dev)
    hc = torch.view_as_complex(torch.full((F, U, A, K, 2), nan, device=dev))
    llr = torch.full((F, D, U, K, b), nan, device=dev) if soft else None
    sinr = torch.full((F, U, K), nan, device=dev) if soft else None
    d_rx = _to_dev(rx)
    torch.cuda.synchronize()
    if soft:
        bad = r.demod_frames_device_mu_soft(d_rx, F, U, comb, llr, bits, hc, sinr, detector=detector, noise_var=noise_var,
                                            count_singular=count)
    else:
        bad = r.demod_frames_device_mu(d_rx, F, U, comb, bits, hc, detector=detector, noise_var=noise_var, count_singular=count)
    r.sync()
    out = {"combined": comb.cpu().numpy(), "bits": bits.cpu().numpy(), "hconj": hc.cpu().numpy(), "n_singular": bad}
    if soft:
        out["llr"] = llr.cpu().numpy()
        out["sinr"] = sinr.cpu().numpy()
    return out


COMB_CASES = [  # (A, N, C, S, U, detector, b): every plan from 64 to 4096 points
    (4, 64, 16, 6, 2, "zf", 2),
    (16, 64, 16, 5, 16, "zf", 2),          # 16 users on 63 subcarriers: 3-4 pilots each
    (16, 64, 16, 5, 16, "mmse", 4),
    (8, 128, 16, 6, 4, "mmse", 4),
    (32, 256, 32, 6, 4, "zf", 4),
    (32, 512, 32, 6, 8, "mmse", 6),
    (64, 1024, 64, 8, 8, "zf", 4),
    (64, 1024, 64, 8, 16, "mmse", 4),
    (128, 2048, 144, 6, 8, "zf", 6),
    (64, 4096, 288, 5, 4, "mmse", 4),
    (256, 4096, 288, 14, 16, "zf", 6),     # c4 with 16 users in 14 symbols: impossible with time-orthogonal pilots
]
_CASE_ID = "A{}_N{}_C{}_S{}_U{}_{}_b{}"


@pytest.mark.gpu
@pytest.mark.parametrize("case", COMB_CASES, ids=lambda c: _CASE_ID.format(*c))
def test_gpu_matches_comb_ref(ofdm, case):
    A, N, C, S, U, det, b = case
    F = 2
    nv = 0.02 if det == "mmse" else 0.0
    d = comb_frames(F, A, N, C, S, b, U, 30.0, seed=A + N + U)
    ref = comb_ref(d["rx"], d["pilot_asc"], C, U, nv, b)
    assert ref["n_singular"] == 0
    with ofdm.LsMrcReceiver(A, N, C, S, b) as r:
        r.set_pilot(d["pilot_asc"])
        r.set_mu_pilots("comb")
        got = _run(r, d["rx"], F, U, b, det, nv, count=True)
    assert got["n_singular"] == 0
    assert_close(got["hconj"], ref["hconj"], "hconj")
    tol = max(1e-5, 4e-6 * ref["gram_cond"])
    assert_close(got["combined"], ref["combined"], "combined", tol=tol)
    assert_bits_match(got["bits"], ref["bits"], ref["combined"], b, "bits", got["combined"], tol=tol)


@pytest.mark.gpu
@pytest.mark.parametrize("N,C", [(64, 16), (128, 16), (256, 32), (512, 32), (1024, 64), (2048, 144), (4096, 288)])
def test_gpu_own_pilots_are_the_single_user_estimate(ofdm, N, C):
    """On user u's comb, the exported conj(H) is the single-user pilot launch's, bit for bit."""
    import torch

    A, S, b, U, F = 8, 4, 4, 5, 3
    K = N - 1
    d = comb_frames(F, A, N, C, S, b, U, 25.0, seed=N)
    with ofdm.LsMrcReceiver(A, N, C, S, b) as r:
        r.set_pilot(d["pilot_asc"])
        r.set_oneshot(0)
        d_rx = _to_dev(d["rx"])
        comb = torch.zeros((F, S - 1, K), dtype=torch.complex64, device=_dev())
        hc = torch.zeros((F, A, K), dtype=torch.complex64, device=_dev())
        torch.cuda.synchronize()
        r.demod_frames_device(d_rx, F, comb, None, hc)
        r.sync()
        su = hc.cpu().numpy()
        r.set_mu_pilots("comb")
        mu = _run(r, d_rx, F, U, b)["hconj"]
    synth = ofdm.synth
    su_asc, mu_asc = synth.bin_to_asc(su), synth.bin_to_asc(mu)
    for u in range(U):
        assert mu_asc[:, u, :, u::U].tobytes() == su_asc[:, :, u::U].tobytes(), u


@pytest.mark.gpu
@pytest.mark.parametrize("N,C", [(64, 16), (128, 16), (256, 32), (512, 32), (1024, 64), (2048, 144), (4096, 288)])
def test_gpu_single_user_comb_is_time(ofdm, N, C):
    A, S, b, F = 8, 5, 4, 3
    nv = noise_var_of(20.0, N)
    d = ofdm.synth.make_frames_mu(F, A, N, C, S, b, 1, snr_db=20.0, seed=N + 1)
    with ofdm.LsMrcReceiver(A, N, C, S, b) as r:
        r.set_pilot(d["pilot_asc"])
        runs = {}
        for layout in ("time", "comb"):
            r.set_mu_pilots(layout)
            runs[layout] = [_run(r, d["rx"], F, 1, b, det, nv, soft=soft) for det in ("zf", "mmse") for soft in (False, True)]
    for t, c in zip(runs["time"], runs["comb"]):
        for key in t:
            if key != "n_singular":
                assert t[key].tobytes() == c[key].tobytes(), key


@pytest.mark.gpu
def test_gpu_noiseless_flat_channel_decodes_exactly(ofdm):
    A, N, C, S, U, b, F = 16, 256, 32, 6, 8, 6, 2
    d = comb_frames(F, A, N, C, S, b, U, None, seed=5, n_taps=1)
    with ofdm.LsMrcReceiver(A, N, C, S, b) as r:
        r.set_pilot(d["pilot_asc"])
        r.set_mu_pilots("comb")
        got = _run(r, d["rx"], F, U, b)
    assert np.array_equal(got["bits"], ofdm.synth.pack_bits_rows(d["src_idx"], b))


@pytest.mark.gpu
@pytest.mark.parametrize("case", DECODE_CASES, ids=lambda c: "A{}_N{}_U{}".format(c[0], c[1], c[4]))
def test_gpu_multipath_30db_decodes_error_free(ofdm, case):
    A, N, C, S, U, b, snr, seed, L = case
    F = 2
    d = comb_frames(F, A, N, C, S, b, U, snr, seed, n_taps=L)
    with ofdm.LsMrcReceiver(A, N, C, S, b) as r:
        r.set_pilot(d["pilot_asc"])
        r.set_mu_pilots("comb")
        got = _run(r, d["rx"], F, U, b)
        again = _run(r, d["rx"], F, U, b)
    assert np.array_equal(got["bits"], ofdm.synth.pack_bits_rows(d["src_idx"], b))
    assert got["combined"].tobytes() == again["combined"].tobytes() and got["bits"].tobytes() == again["bits"].tobytes()


@pytest.mark.gpu
@pytest.mark.parametrize("det,b", [("zf", 4), ("mmse", 6), ("zf", 2)])
@pytest.mark.parametrize("A,N,C,S,U", [(32, 1024, 64, 5, 8), (16, 64, 16, 4, 16), (64, 4096, 288, 4, 4)])
def test_gpu_soft_comb_call(ofdm, det, b, A, N, C, S, U):
    F, snr = 2, 20.0
    nv = noise_var_of(snr, N)
    d = comb_frames(F, A, N, C, S, b, U, snr, seed=N + U + b)
    ref = comb_ref(d["rx"], d["pilot_asc"], C, U, nv if det == "mmse" else 0.0, b)
    assert ref["n_singular"] == 0
    want = soft_ref(ref, det, nv, b)
    with ofdm.LsMrcReceiver(A, N, C, S, b) as r:
        r.set_pilot(d["pilot_asc"])
        r.set_mu_pilots("comb")
        hard = _run(r, d["rx"], F, U, b, det, nv)
        soft = _run(r, d["rx"], F, U, b, det, nv, soft=True)
    K = N - 1
    assert soft["llr"].shape == (F, S - 1, U, K, b) and soft["sinr"].shape == (F, U, K)
    assert soft["combined"].tobytes() == hard["combined"].tobytes() and soft["bits"].tobytes() == hard["bits"].tobytes()
    assert np.isfinite(soft["llr"]).all() and np.isfinite(soft["sinr"]).all()
    tol = max(2e-5, 4e-6 * ref["gram_cond"])
    err = llr_row_err(soft["llr"], want["llr"])
    assert err.max() <= tol, (err.max(), tol)
    s_err = np.abs(soft["sinr"] - want["sinr"]).max(-1) / want["sinr"].max(-1)
    assert s_err.max() <= tol, (s_err.max(), tol)


@pytest.mark.gpu
def test_gpu_downlink_loop_back_from_the_comb_estimate(ofdm):
    """Comb uplink -> exported conj(H) -> lsmrc_precode_frames_device -> the library's FFT of tx -> each user's true
    channel: every user recovers its bits at 30 dB on a multipath channel."""
    import torch

    A, N, C, S, U, b, snr, seed, L = LOOPBACK_CASE
    F, Sd, K = 2, 3, N - 1
    synth = ofdm.synth
    dev = _dev()
    rng = np.random.default_rng(seed + 1)
    idx = rng.integers(0, 1 << b, size=(F, Sd, U, K), dtype=np.uint8)
    sym = synth.qam_map_indices(idx, b).astype(np.complex64)
    up = comb_frames(F, A, N, C, S, b, U, snr, seed, n_taps=L)
    with ofdm.LsMrcReceiver(A, N, C, S, b) as r:
        r.set_pilot(up["pilot_asc"])
        r.set_mu_pilots("comb")
        hc = torch.from_numpy(_run(r, up["rx"], F, U, b)["hconj"]).to(dev)
        tx = torch.zeros((F, Sd, A, N + C), dtype=torch.complex64, device=dev)
        gain = torch.zeros((F,), dtype=torch.float32, device=dev)
        torch.cuda.synchronize()
        assert r.precode_frames_device(hc, F, U, torch.from_numpy(sym).to(dev), Sd, tx, gain, count_singular=True) == 0
        rows = torch.empty((F, Sd, A, N), dtype=torch.complex64, device=dev)
        r.stage("drop_prefix", rows, tx, F * Sd * A)
        r.stage("fft", rows, F * Sd * A)
        r.sync()
        y = rows.cpu().numpy().astype(np.complex128)
        g = gain.cpu().numpy().astype(np.float64)
    rx_user = np.einsum("fuak,fdak->fduk", up["h_true"], y[..., 1:]) / g[:, None, None, None]
    assert np.array_equal(demap(synth.bin_to_asc(rx_user), b), idx), "bit errors at 30 dB"


@pytest.mark.gpu
def test_gpu_singular_subcarriers(ofdm):
    """Users 0 and 1 share one flat channel in frame 0: every subcarrier of that frame is singular; frame 1 is regular."""
    A, N, C, S, U, b, F = 8, 256, 32, 4, 3, 4, 2
    K = N - 1
    h = ofdm.synth.multipath_channel(F, U, A, N, 1, seed=6)
    h[0, 1] = h[0, 0]
    d = comb_frames(F, A, N, C, S, b, U, None, seed=6, h=h)
    ref = comb_ref(d["rx"], d["pilot_asc"], C, U, 0.0, b)
    assert ref["n_singular"] == K and ref["singular"][0].all()
    with ofdm.LsMrcReceiver(A, N, C, S, b) as r:
        r.set_pilot(d["pilot_asc"])
        r.set_mu_pilots("comb")
        got = _run(r, d["rx"], F, U, b, count=True)
        mm = _run(r, d["rx"], F, U, b, "mmse", 0.1, count=True)
    assert got["n_singular"] == ref["n_singular"]
    assert not got["combined"][0].any()
    assert_close(got["combined"][1], ref["combined"][1], "combined", tol=max(1e-5, 4e-6 * ref["gram_cond"]))
    assert mm["n_singular"] == 0 and np.isfinite(mm["combined"].view(np.float32)).all()


@pytest.mark.gpu
def test_gpu_layout_switching_on_one_handle(ofdm):
    A, N, C, S, b, F = 16, 1024, 64, 8, 4, 2
    tf = ofdm.synth.make_frames_mu(F, A, N, C, S, b, 4, snr_db=25.0, seed=7)
    cf = comb_frames(F, A, N, C, S, b, 6, 25.0, seed=8, h=ofdm.synth.multipath_channel(F, 6, A, N, 4, seed=8))
    cf = ofdm.synth.make_frames_mu(F, A, N, C, S, b, 6, snr_db=25.0, seed=8, pilot_asc=tf["pilot_asc"], h=cf["h_true"],
                                   pilots="comb")
    with ofdm.LsMrcReceiver(A, N, C, S, b) as r:
        r.set_pilot(tf["pilot_asc"])
        t0 = _run(r, tf["rx"], F, 4, b, P=4)                                  # default layout: time
        r.set_mu_pilots("time")
        t1 = _run(r, tf["rx"], F, 4, b, P=4)
        r.set_mu_pilots("comb")
        c0 = _run(r, cf["rx"], F, 6, b)
        c1 = _run(r, cf["rx"], F, 6, b, soft=True, noise_var=0.01)
        r.set_mu_pilots("time")
        t2 = _run(r, tf["rx"], F, 4, b, P=4)
        r.set_mu_pilots("comb")
        c2 = _run(r, cf["rx"], F, 6, b)
        for bad in (2, -1, 7):
            with pytest.raises(ofdm.LsmrcError) as e:
                r._ck(r.lib.lsmrc_set_mu_pilots(r.h, bad))
            assert e.value.code == -1
        with pytest.raises(ofdm.LsmrcError):
            r.set_mu_pilots("dft")
        c3 = _run(r, cf["rx"], F, 6, b)                                       # a rejected value left the layout alone
    for x in (t1, t2):
        assert all(x[k].tobytes() == t0[k].tobytes() for k in ("combined", "bits", "hconj"))
    for x in (c1, c2, c3):
        assert all(x[k].tobytes() == c0[k].tobytes() for k in ("combined", "bits", "hconj"))
    ref = comb_ref(cf["rx"], tf["pilot_asc"], C, 6, 0.0, b)
    assert_close(c0["combined"], ref["combined"], "combined", tol=max(1e-5, 4e-6 * ref["gram_cond"]))


@pytest.mark.gpu
@pytest.mark.parametrize("soft", [False, True], ids=["hard", "soft"])
@pytest.mark.parametrize("dims", [(8, 64, 16, 3, 2, 6), (32, 1024, 64, 4, 4, 8), (64, 4096, 288, 3, 4, 4)])
def test_gpu_comb_call_replays_from_a_cuda_graph(ofdm, soft, dims):
    """Captured in comb mode, the graph keeps comb pilots even after the handle is switched back to time."""
    import torch

    A, N, C, S, b, U = dims
    F, K = 2, N - 1
    dev = _dev()
    user = torch.cuda.Stream(dev)
    g = torch.Generator(device=dev).manual_seed(11)
    inputs = [torch.randn((F, S, A, N + C, 2), device=dev, generator=g) for _ in range(3)]
    rx = torch.empty_like(inputs[0])
    comb = torch.zeros((F, S - 1, U, K, 2), device=dev)
    bits = torch.zeros((F, S - 1, U, (K * b + 7) // 8), device=dev, dtype=torch.uint8)
    hc = torch.zeros((F, U, A, K, 2), device=dev)
    llr = torch.zeros((F, S - 1, U, K, b), device=dev)
    sinr = torch.zeros((F, U, K), device=dev)
    outs = (comb, bits, hc, llr, sinr) if soft else (comb, bits, hc)
    torch.cuda.synchronize(dev)
    with ofdm.LsMrcReceiver(A, N, C, S, b) as r:
        r.set_pilot(ofdm.synth.make_pilot(K, 3))
        r.set_stream(user.cuda_stream)
        r.set_mu_pilots("comb")

        def call():
            if soft:
                r.demod_frames_device_mu_soft(rx, F, U, comb, llr, bits, hc, sinr, detector="mmse", noise_var=0.1)
            else:
                r.demod_frames_device_mu(rx, F, U, comb, bits, hc, detector="mmse", noise_var=0.1)

        with torch.cuda.stream(user):
            rx.copy_(inputs[0])
            call()                                  # first call: scratch allocated outside the capture
        user.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=user):
            call()
        for x in inputs:
            r.set_mu_pilots("time")
            with torch.cuda.stream(user):
                rx.copy_(x)
                for o in outs:
                    o.zero_()
                graph.replay()
            user.synchronize()
            got = [o.clone() for o in outs]
            r.set_mu_pilots("comb")
            with torch.cuda.stream(user):
                for o in outs:
                    o.zero_()
                call()
            user.synchronize()
            assert all(torch.equal(a, o) for a, o in zip(got, outs))
            assert bool(torch.isfinite(comb).all()) and float(comb.abs().max()) > 0
        r.set_stream(None)


@pytest.mark.gpu
def test_gpu_more_frames_than_one_grid_dimension(ofdm):
    """65537 frames: every frame is decoded as in a small call."""
    import torch

    A, N, C, S, U, b, F = 4, 64, 16, 3, 4, 2, 65537
    K = N - 1
    dev = _dev()
    d = comb_frames(4, A, N, C, S, b, U, 30.0, seed=65)
    small = _to_dev(d["rx"])
    big = small[torch.arange(F, device=dev) % 4].contiguous()
    with ofdm.LsMrcReceiver(A, N, C, S, b) as r:
        r.set_pilot(d["pilot_asc"])
        r.set_mu_pilots("comb")
        want = _run(r, small, 4, U, b)
        comb = torch.zeros((F, S - 1, U, K), dtype=torch.complex64, device=dev)
        bits = torch.zeros((F, S - 1, U, (K * b + 7) // 8), dtype=torch.uint8, device=dev)
        hc = torch.zeros((F, U, A, K), dtype=torch.complex64, device=dev)
        torch.cuda.synchronize()
        assert r.demod_frames_device_mu(big, F, U, comb, bits, hc, count_singular=True) == 0
        for f in (0, 3, 65532, 65535, 65536):
            assert comb[f].cpu().numpy().tobytes() == want["combined"][f % 4].tobytes(), f
            assert bits[f].cpu().numpy().tobytes() == want["bits"][f % 4].tobytes(), f
            assert hc[f].cpu().numpy().tobytes() == want["hconj"][f % 4].tobytes(), f
        whole = comb[:65536].view(16384, 4, S - 1, U, K)
        assert bool((whole == torch.from_numpy(want["combined"]).to(dev)).all())
        wh = hc[:65536].view(16384, 4, U, A, K)
        assert bool((wh == torch.from_numpy(want["hconj"]).to(dev)).all())


@pytest.mark.gpu
def test_gpu_argument_errors(ofdm):
    import torch

    dev = _dev()
    N, C, b = 64, 16, 2
    K = N - 1
    # comb accepts U >= S; time still rejects it
    A, S = 8, 3
    d = comb_frames(1, A, N, C, S, b, 6, 30.0, seed=9)
    rx = _to_dev(d["rx"])
    comb = torch.zeros((1, S - 1, 6, K), dtype=torch.complex64, device=dev)
    with ofdm.LsMrcReceiver(A, N, C, S, b) as r:
        r.set_pilot(d["pilot_asc"])
        n0 = r.launch_count()
        with pytest.raises(ofdm.LsmrcError) as e:
            r.demod_frames_device_mu(rx, 1, 6, comb)                           # default: time pilots, U >= S
        assert e.value.code == -1 and r.launch_count() == n0
        r.set_mu_pilots("comb")
        torch.cuda.synchronize()
        r.demod_frames_device_mu(rx, 1, 6, comb)
        r.sync()
        assert r.launch_count() > n0
        n1 = r.launch_count()
        for U in (0, 9, 17):                                                   # U > A = 8, U > 16
            with pytest.raises(ofdm.LsmrcError) as e:
                r.demod_frames_device_mu(rx, 1, U, comb)
            assert e.value.code == -1, U
            with pytest.raises(ofdm.LsmrcError) as e:
                r.demod_frames_device_mu_soft(rx, 1, U, comb, comb, noise_var=0.1)
            assert e.value.code == -1, U
        assert r.launch_count() == n1
    with ofdm.LsMrcReceiver(32, N, C, S, b) as r:
        r.set_pilot(d["pilot_asc"])
        r.set_mu_pilots("comb")
        n0 = r.launch_count()
        with pytest.raises(ofdm.LsmrcError) as e:
            r.demod_frames_device_mu(rx, 1, 17, comb)
        assert e.value.code == -1 and r.launch_count() == n0
    with ofdm.LsMrcReceiver(A, N, C, 1, b) as r:                              # S = 1: no symbol left for data
        r.set_pilot(d["pilot_asc"])
        r.set_mu_pilots("comb")
        n0 = r.launch_count()
        for U in (1, 2):
            with pytest.raises(ofdm.LsmrcError) as e:
                r.demod_frames_device_mu(rx, 1, U, comb)
            assert e.value.code == -1
        assert r.launch_count() == n0
