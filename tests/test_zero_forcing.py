"""Multi-user zero-forcing helpers (SURVEY 8f rank 4; cpuLS.hpp:400-463 -- defined but uncalled in the reference, and
built on CBLAS/LAPACK which are absent here: parity unpinned).  The oracle restates the call sequence; both the
oracle and the CUDA kernels are checked against the defining property  Xk * Hk = I  and against each other."""
import numpy as np
import pytest


def _channels(U, A, K, seed):
    rng = np.random.default_rng(seed)
    return ((rng.standard_normal((U, A, K)) + 1j * rng.standard_normal((U, A, K))) / np.sqrt(2)).astype(np.complex64)


@pytest.mark.parametrize("U,A,K", [(1, 1, 7), (2, 4, 63), (4, 16, 255), (16, 16, 31)])
def test_oracle_zero_forcing_inverts_the_channel(oracle, U, A, K):
    X = _channels(U, A, K, 1)
    H, bad = oracle.zf_create(X)
    assert bad == 0 and H.shape == (K, U, A)
    cond = max(np.linalg.cond(X[:, :, k].astype(np.complex128)) for k in range(K))
    for k in range(K):
        assert np.abs(X[:, :, k].astype(np.complex128) @ H[k].T - np.eye(U)).max() < 2e-6 * cond * cond
    # against the textbook right inverse in double precision
    k = K // 2
    Xk = X[:, :, k].astype(np.complex128)
    want = Xk.conj().T @ np.linalg.inv(Xk @ Xk.conj().T)
    assert np.abs(H[k].T - want).max() < 2e-6 * cond * cond * np.abs(want).max()
    # precoded symbols arrive interference-free: Xk * (Hk xd) = xd
    xd = _channels(1, U, K, 2)[0]
    hx = oracle.zf_apply(H, xd)
    got = np.stack([X[:, :, k].astype(np.complex128) @ hx[:, k] for k in range(K)], axis=1)
    assert np.abs(got - xd).max() < 1e-5 * cond * cond


def test_oracle_flags_singular_subcarriers(oracle):
    X = _channels(2, 4, 9, 3)
    X[1, :, 4] = X[0, :, 4]          # two identical users on subcarrier 4
    H, bad = oracle.zf_create(X)
    assert bad == 1 and not H[4].any() and H[3].any()


@pytest.mark.gpu
@pytest.mark.parametrize("U,A,K", [(1, 1, 7), (2, 4, 63), (4, 64, 1023), (8, 32, 100), (16, 16, 31), (4, 256, 4095),
                                   (3, 8, 63), (5, 16, 255), (7, 32, 100), (9, 24, 1023),
                                   (15, 256, 4095)])   # (15 users on 256 antennas: 4 subcarriers per CTA, the last CTA 3)
def test_gpu_zero_forcing_matches_oracle(ofdm, oracle, U, A, K):
    import torch

    X = _channels(U, A, K, 5)
    xd = _channels(1, U, K, 6)[0]
    want_h, _ = oracle.zf_create(X)
    want_hx = oracle.zf_apply(want_h, xd)
    dev = torch.device("cuda:0")
    dx = torch.view_as_real(torch.from_numpy(X).to(dev)).contiguous()
    dxd = torch.view_as_real(torch.from_numpy(xd).to(dev)).contiguous()
    dh = torch.full((K, U, A, 2), float("nan"), device=dev)
    dhx = torch.full((A, K, 2), float("nan"), device=dev)
    with ofdm.LsMrcReceiver(4, 64, 16, 4, 2) as r:      # the ZF helpers do not depend on the receiver's dimensions
        assert r.zf_create(dx, A, K, U, dh) == 0
        r.zf_apply(dh, dxd, A, K, U, dhx)
        r.sync()
        with pytest.raises(ofdm.LsmrcError):
            r.zf_create(dx, 2, K, 3, dh)                # more users than antennas
    got_h = torch.view_as_complex(dh).cpu().numpy()
    got_hx = torch.view_as_complex(dhx).cpu().numpy()
    cond = max(np.linalg.cond(X[:, :, k].astype(np.complex128)) for k in range(0, K, max(1, K // 64)))
    tol = 4e-6 * cond * cond
    assert np.isfinite(got_h.view(np.float32)).all()
    assert np.abs(got_h - want_h).max() <= tol * np.abs(want_h).max(), (np.abs(got_h - want_h).max(), cond)
    assert np.abs(got_hx - want_hx).max() <= tol * np.abs(want_hx).max()
    for k in range(0, K, max(1, K // 16)):
        assert np.abs(X[:, :, k].astype(np.complex128) @ got_h[k].T - np.eye(U)).max() < tol


@pytest.mark.gpu
def test_gpu_zero_forcing_counts_singular_subcarriers(ofdm):
    import torch

    X = _channels(2, 4, 9, 3)
    X[1, :, 4] = X[0, :, 4]
    dev = torch.device("cuda:0")
    dx = torch.view_as_real(torch.from_numpy(X).to(dev)).contiguous()
    dh = torch.full((9, 2, 4, 2), float("nan"), device=dev)
    with ofdm.LsMrcReceiver(4, 64, 16, 4, 2) as r:
        bad = r.zf_create(dx, 4, 9, 2, dh)
    h = torch.view_as_complex(dh).cpu().numpy()
    assert bad == 1 and not h[4].any()
    assert np.isfinite(h[[0, 1, 2, 3, 5, 6, 7, 8]].view(np.float32)).all()


@pytest.mark.parametrize("U,A,K", [(2, 4, 63), (4, 16, 255), (4, 64, 1023), (8, 32, 64)])
def test_oracle_equals_the_reference_call_sequence_on_real_lapack(oracle, U, A, K):
    """Pin for this row: createZeroForcingMatrix / multiplyWithChannelInv (cpuLS.hpp:415-463) call cblas_cgemm,
    cgetrf_, cgetri_ and cblas_cgemv in complex64.  CBLAS/LAPACK headers are absent from this image, so the reference
    function cannot be compiled -- but scipy ships the very same routines (OpenBLAS): the reference's call sequence is
    replayed here on them, per subcarrier, in complex64, and the oracle (plain loops + Gauss-Jordan in double) must agree
    to single-precision rounding amplified by the conditioning of the Gram matrix."""
    from scipy.linalg import blas, lapack

    X = _channels(U, A, K, 11)
    xd = _channels(1, U, K, 12)[0]
    got_h, bad = oracle.zf_create(X)
    got_hx = oracle.zf_apply(got_h, xd)
    assert bad == 0
    one = np.complex64(1)
    want_h = np.empty((K, U, A), np.complex64)
    want_hx = np.empty((A, K), np.complex64)
    worst = 0.0
    for k in range(K):
        Xk = np.asfortranarray(X[:, :, k])                       # rotCube: users x rows, column-major, ld = users
        G = blas.cgemm(one, Xk, Xk, trans_b=2)                   # Xk * Xk^H                 (cpuLS.hpp:437)
        lu, piv, info = lapack.cgetrf(G)                         #                            (:438)
        assert info == 0
        Ginv, info = lapack.cgetri(lu, piv)                      #                            (:439)
        assert info == 0
        Hk = blas.cgemm(one, Xk, Ginv, trans_a=2)                # Xk^H * inv, rows x users   (:440)
        want_h[k] = Hk.T                                         # stored column-major with ld = rows: H[k][u][a]
        want_hx[:, k] = blas.cgemv(one, Hk, xd[:, k])            # multiplyWithChannelInv     (:460)
        worst = max(worst, np.linalg.cond(G.astype(np.complex128)))
    tol = 3e-6 * worst
    assert np.abs(got_h - want_h).max() <= tol * np.abs(want_h).max(), (np.abs(got_h - want_h).max() / np.abs(want_h).max(), worst)
    assert np.abs(got_hx - want_hx).max() <= tol * np.abs(want_hx).max()
