"""Float64 references of the multi-user calls, shared by the multi-user test files.  Plain numpy -- CP strip,
np.fft.fft, LS estimate, np.linalg.solve per subcarrier, hard decisions -- independent of the library and of the C
oracles:
  mu_ref64     the uplink (lsmrc_demod_frames_device_mu) with time-orthogonal or comb pilots;
  comb_ref     its comb-pilot branch (the interpolation rule interp_comb);
  soft_ref     SINR and max-log LLRs of the soft call (lsmrc_demod_frames_device_mu_soft) on top of either;
  precode_ref  the downlink (lsmrc_precode_frames_device)."""
import numpy as np

SINGULAR_COND = 1e8  # a Gram matrix this badly conditioned in float64 is singular (the tests make such ones exactly)
A_EXACT = {2: 1 / np.sqrt(2.0), 4: 1 / np.sqrt(10.0), 6: 1 / np.sqrt(42.0)}


def _synth():
    from gpu_accel_ofdm_ls_mrc_b200 import synth

    return synth


def _asc_to_bin(v):
    from gpu_accel_ofdm_ls_mrc_b200.synth import asc_to_bin

    return asc_to_bin(v)


def phi(i, N):
    """signed frequency of ascending index i (DC skipped)"""
    i = np.asarray(i)
    return np.where(i < N // 2, i - N // 2, i - N // 2 + 1)


def interp_comb(ls_asc, U, N):
    """The comb rule on ascending-frequency LS values ls_asc [..., K] (float64): [..., U, K], user u copied on its own
    pilots i = u mod U, linear in phi between its two nearest pilots, the nearest pilot held beyond its outermost ones."""
    ls_asc = np.asarray(ls_asc).astype(np.complex128)
    K = ls_asc.shape[-1]
    i = np.arange(K)
    ph = phi(i, N).astype(np.float64)
    out = np.empty(ls_asc.shape[:-1] + (U, K), np.complex128)
    for u in range(U):
        own = np.arange(u, K, U)
        j = np.clip(np.searchsorted(own, i, side="right") - 1, 0, len(own) - 1)
        p0 = own[j]
        p1 = own[np.minimum(j + 1, len(own) - 1)]
        inside = (i > p0) & (p1 > p0)
        w = np.where(inside, (ph - ph[p0]) / np.where(inside, ph[p1] - ph[p0], 1.0), 0.0)
        a, b = ls_asc[..., p0], ls_asc[..., p1]
        out[..., u, :] = np.where(inside, a + w * (b - a), a)
    return out


def demap(y, b):
    """nearest constellation point of the Gray-mapped QAM (synth.qam_map_indices) per axis -> symbol index"""
    synth = _synth()
    pts = synth.qam_map_indices(np.arange(1 << b), b)
    lv = np.unique(np.round(pts.real, 12))
    m = len(lv)
    table = np.zeros((m, m), np.uint8)
    table[np.searchsorted(lv, np.round(pts.real, 12)), np.searchsorted(lv, np.round(pts.imag, 12))] = np.arange(1 << b)
    step = lv[1] - lv[0]
    ri = np.clip(np.rint((y.real - lv[0]) / step), 0, m - 1).astype(np.int64)
    ii = np.clip(np.rint((y.imag - lv[0]) / step), 0, m - 1).astype(np.int64)
    return table[ri, ii]


def comb_ref(rx, pilot_asc, C, U, lam, b=None):
    """rx [F,S,A,N+C] comb frames -> dict(hconj [F,U,A,K] conj(H) bin order, combined [F,S-1,U,K] ascending frequency,
    bits [F,S-1,U,row] (with b), ginv_diag [F,U,K] bin order, singular [F,K] bin order, gram_cond (over the regular
    subcarriers)).  Singular subcarriers (cond > SINGULAR_COND) get W = 0."""
    synth = _synth()
    rx = np.asarray(rx)
    N = rx.shape[-1] - C
    z = np.fft.fft(rx[..., C:].astype(np.complex128), axis=-1)[..., 1:]          # [F,S,A,K] bin order
    x_bin = synth.asc_to_bin(np.asarray(pilot_asc).astype(np.complex128))
    ls = np.conj(z[:, 0] / x_bin)                                                # [F,A,K] as the pilot kernel exports it
    hc = interp_comb(synth.bin_to_asc(ls), U, N)                                 # [F,A,U,K] ascending
    hconj = synth.asc_to_bin(hc).transpose(0, 2, 1, 3)                           # [F,U,A,K] bin order
    H = np.conj(hconj).transpose(0, 3, 2, 1)                                     # [F,K,A,U]
    Hh = np.conj(np.swapaxes(H, -1, -2))
    G = Hh @ H + lam * np.eye(U)
    cond = np.linalg.cond(G)
    singular = cond > SINGULAR_COND
    Gs = np.where(singular[..., None, None], np.eye(U), G)
    W = np.where(singular[..., None, None], 0.0, np.linalg.solve(Gs, Hh))        # [F,K,U,A]
    M = np.where(singular[..., None, None], 0.0, np.linalg.inv(Gs))
    x = (W @ z[:, 1:].transpose(0, 3, 2, 1)).transpose(0, 3, 2, 1)               # [F,S-1,U,K] bin order
    out = {"hconj": hconj, "combined": synth.bin_to_asc(x), "singular": singular, "n_singular": int(singular.sum()),
           "ginv_diag": np.diagonal(M, axis1=-2, axis2=-1).real.transpose(0, 2, 1),
           "gram_cond": float(np.where(singular, 1.0, cond).max())}
    if b is not None:
        out["bits"] = synth.pack_bits_rows(demap(out["combined"], b), b)
    return out


def mu_ref64(rx, pilot_asc, C, U, lam, b=None, pilots="time"):
    """The multi-user uplink in float64: rx [F,S,A,N+C] -> comb_ref's dict, with P = U pilot symbols (time: user u's
    LS estimate conj(Z[:, u] / X) on symbol u, data in symbols U..S-1) or P = 1 (comb: comb_ref itself); combined and
    bits [F,S-P,U,...].  After the estimate both layouts run the same detector: per subcarrier np.linalg.solve of
    G = H^H H + lam I, W = 0 where cond(G) > SINGULAR_COND, the diagonal of inv(G) and the hard decisions."""
    if pilots == "comb":
        return comb_ref(rx, pilot_asc, C, U, lam, b)
    if pilots != "time":
        raise ValueError(pilots)
    synth = _synth()
    rx = np.asarray(rx)
    z = np.fft.fft(rx[..., C:].astype(np.complex128), axis=-1)[..., 1:]          # [F,S,A,K] bin order
    x_bin = synth.asc_to_bin(np.asarray(pilot_asc).astype(np.complex128))
    hconj = np.conj(z[:, :U] / x_bin)                                            # [F,U,A,K]: user u's pilot is symbol u
    H = np.conj(hconj).transpose(0, 3, 2, 1)                                     # [F,K,A,U]
    Hh = np.conj(np.swapaxes(H, -1, -2))
    G = Hh @ H + lam * np.eye(U)
    cond = np.linalg.cond(G)
    singular = cond > SINGULAR_COND
    Gs = np.where(singular[..., None, None], np.eye(U), G)
    W = np.where(singular[..., None, None], 0.0, np.linalg.solve(Gs, Hh))        # [F,K,U,A]
    M = np.where(singular[..., None, None], 0.0, np.linalg.inv(Gs))
    x = (W @ z[:, U:].transpose(0, 3, 2, 1)).transpose(0, 3, 2, 1)               # [F,S-U,U,K] bin order
    out = {"hconj": hconj, "combined": synth.bin_to_asc(x), "singular": singular, "n_singular": int(singular.sum()),
           "ginv_diag": np.diagonal(M, axis1=-2, axis2=-1).real.transpose(0, 2, 1),
           "gram_cond": float(np.where(singular, 1.0, cond).max())}
    if b is not None:
        out["bits"] = synth.pack_bits_rows(demap(out["combined"], b), b)
    return out


def soft64(y, rho, b):
    """max-log piecewise-linear LLRs (soft_symbol in csrc/lsmrc_kernels.cuh) in float64, exact constants: [..., K, b]"""
    a = A_EXACT[b]
    g = 4 * a * np.asarray(rho, np.float64)
    re, im = y.real, y.imag
    out = [g * re, g * im]
    if b == 4:
        out += [g * (2 * a - np.abs(re)), g * (2 * a - np.abs(im))]
    elif b == 6:
        out += [g * (4 * a - np.abs(re)), g * (4 * a - np.abs(im)),
                g * (2 * a - np.abs(np.abs(re) - 4 * a)), g * (2 * a - np.abs(np.abs(im) - 4 * a))]
    return np.stack(out, axis=-1)


def soft_ref(ref, detector, noise_var, b):
    """DESIGN.md 8f on comb_ref's interpolated H: sinr [F,U,K] and llr [F,S-1,U,K,b], ascending frequency"""
    synth = _synth()
    d = ref["ginv_diag"]
    with np.errstate(divide="ignore", invalid="ignore"):
        if detector == "mmse":
            rho = np.where(d > 0, 1.0 / (noise_var * d) - 1.0, 0.0)
            scale = np.where(rho > 0, 1.0 / (1.0 - noise_var * d), 0.0)
            rho = np.maximum(rho, 0.0)
        else:
            rho = np.where(d > 0, 1.0 / (noise_var * d), 0.0)
            scale = np.where(d > 0, 1.0, 0.0)
    rho, scale = synth.bin_to_asc(rho), synth.bin_to_asc(scale)
    y = ref["combined"] * scale[:, None]
    return {"sinr": rho, "llr": soft64(y, rho[:, None, :, :], b)}


def precode_ref(hconj, sym, reg, N, C):
    """hconj [F,U,A,K] conj(H), FFT-bin order; sym [F,Sd,U,K] ascending frequency.  Returns dict(tx [F,Sd,A,N+C] c128,
    gain [F], P [F,K,A,U] (zero on singular subcarriers), singular [F,K] bool)."""
    hconj = np.asarray(hconj).astype(np.complex128)
    F, U, A, K = hconj.shape
    assert K == N - 1
    H = np.conj(hconj).transpose(0, 3, 2, 1)                                 # [F,K,A,U]
    M = np.swapaxes(H, -1, -2) @ np.conj(H) + reg * np.eye(U)                # H^T conj(H) + reg I = conj(G)
    singular = np.linalg.cond(M) > SINGULAR_COND
    M = np.where(singular[..., None, None], np.eye(U), M)
    # P M = conj(H)  <=>  M^T P^T = conj(H)^T
    P = np.swapaxes(np.linalg.solve(np.swapaxes(M, -1, -2), np.swapaxes(np.conj(H), -1, -2)), -1, -2)
    P = np.where(singular[..., None, None], 0.0, P)
    total = (np.abs(P) ** 2).sum(axis=(1, 2, 3))
    gain = np.where(total > 0, np.sqrt(U * K / np.where(total > 0, total, 1.0)), 0.0)
    s_bin = _asc_to_bin(np.asarray(sym).astype(np.complex128))               # [F,Sd,U,K], index k = bin k+1
    z = np.zeros(s_bin.shape[:2] + (A, N), np.complex128)
    z[..., 1:] = np.einsum("fkau,fduk->fdak", P, s_bin)
    t = gain[:, None, None, None] * np.fft.ifft(z, axis=-1)
    tx = np.concatenate([t[..., N - C:], t], axis=-1) if C > 0 else t
    return {"tx": tx, "gain": gain, "P": P, "singular": singular, "z": z}
