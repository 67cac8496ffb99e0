"""Synthetic uplink frames (the reference ships no data and no generator; SURVEY.md 8d).

Per frame: seeded QAM source bits -> Gray-mapped unit-power constellation on bins
1..N-1 (bin 0 = DC left empty, as the receiver drops it: cpuLS.hpp:292,355), a fixed
unit-modulus QPSK pilot as symbol 0, block-fading i.i.d. Rayleigh channel per antenna
and subcarrier, IFFT, cyclic prefix, AWGN at the configured per-antenna SNR.
Layout [F][S][A][N+C] complex64 -- ring-slot order (ShMemSymBuff.hpp:92-106).

numpy version for the CPU-sized parity tests, torch version to build full-size
batches directly in HBM.  Used to feed the receiver; not part of the receive path.
"""
from __future__ import annotations

import numpy as np

_QAM_SCALE = {2: np.sqrt(2.0), 4: np.sqrt(10.0), 6: np.sqrt(42.0)}


def qam_map_indices(idx: np.ndarray, qam_bits: int) -> np.ndarray:
    """3GPP TS 38.211 5.1.3-5.1.5 mapping; idx holds b bits, bit j = b_j (LSB first)."""
    idx = np.asarray(idx).astype(np.int64)
    b = [(idx >> j) & 1 for j in range(qam_bits)]
    if qam_bits == 2:
        re = 1 - 2 * b[0]
        im = 1 - 2 * b[1]
    elif qam_bits == 4:
        re = (1 - 2 * b[0]) * (2 - (1 - 2 * b[2]))
        im = (1 - 2 * b[1]) * (2 - (1 - 2 * b[3]))
    elif qam_bits == 6:
        re = (1 - 2 * b[0]) * (4 - (1 - 2 * b[2]) * (2 - (1 - 2 * b[4])))
        im = (1 - 2 * b[1]) * (4 - (1 - 2 * b[3]) * (2 - (1 - 2 * b[5])))
    else:
        raise ValueError("qam_bits must be 2, 4 or 6")
    return (re + 1j * im) / _QAM_SCALE[qam_bits]


def make_pilot(K: int, seed: int) -> np.ndarray:
    """Unit-modulus QPSK pilot, ascending-frequency order (the Pilots.dat order)."""
    rng = np.random.default_rng(seed ^ 0x5EED)
    return np.exp(1j * (np.pi / 4) * (2 * rng.integers(0, 4, K) + 1)).astype(np.complex64)


def asc_to_bin(v_asc: np.ndarray) -> np.ndarray:
    """ascending frequency [bin N/2..N-1, 1..N/2-1] -> FFT-bin order [1..N-1] (last axis)."""
    K = v_asc.shape[-1]
    return np.roll(v_asc, -((K + 1) // 2), axis=-1)


def bin_to_asc(v_bin: np.ndarray) -> np.ndarray:
    K = v_bin.shape[-1]
    return np.roll(v_bin, (K + 1) // 2, axis=-1)


def pack_bits_rows(idx: np.ndarray, qam_bits: int) -> np.ndarray:
    """idx [..., K] symbol indices -> packed rows [..., ceil(K*b/8)], LSB first."""
    idx = np.asarray(idx, dtype=np.uint8)
    K = idx.shape[-1]
    bits = ((idx[..., None] >> np.arange(qam_bits, dtype=np.uint8)) & 1).reshape(*idx.shape[:-1], K * qam_bits)
    return np.packbits(bits, axis=-1, bitorder="little")


def make_frames(n_frames, n_ant, fft_size, cp_len, n_sym, qam_bits, snr_db=None, seed=0,
                channel="rayleigh", pilot_asc=None):
    """Returns dict(rx [F,S,A,N+C] c64, pilot_asc [K] c64, src_idx [F,S-1,K] u8 (ascending
    frequency), h_true [F,A,K] c128 (bin order))."""
    F, A, N, C, S = n_frames, n_ant, fft_size, cp_len, n_sym
    K = N - 1
    rng = np.random.default_rng(seed)
    pilot_asc = make_pilot(K, seed) if pilot_asc is None else np.asarray(pilot_asc, np.complex64)
    src_idx = rng.integers(0, 1 << qam_bits, size=(F, S - 1, K), dtype=np.uint8)
    data_asc = qam_map_indices(src_idx, qam_bits)
    tx_bin = np.zeros((F, S, N), np.complex128)
    tx_bin[:, 0, 1:] = asc_to_bin(pilot_asc.astype(np.complex128))
    tx_bin[:, 1:, 1:] = asc_to_bin(data_asc)
    if channel == "identity":
        h = np.ones((F, A, K), np.complex128)
    elif channel == "unit":  # unit modulus, random phase: no deep fades (for single-antenna cases)
        h = np.exp(2j * np.pi * rng.random((F, A, K)))
    else:
        h = (rng.standard_normal((F, A, K)) + 1j * rng.standard_normal((F, A, K))) / np.sqrt(2.0)
    hfull = np.zeros((F, A, N), np.complex128)
    hfull[:, :, 1:] = h
    yf = tx_bin[:, :, None, :] * hfull[:, None, :, :]          # [F,S,A,N]
    yt = np.fft.ifft(yf, axis=-1)                               # unnormalised forward FFT undoes this
    if snr_db is not None:
        sig_pow = K / (N * N)                                   # per time sample, unit-power bins
        sigma = np.sqrt(sig_pow / (10.0 ** (snr_db / 10.0)) / 2.0)
        yt = yt + sigma * (rng.standard_normal(yt.shape) + 1j * rng.standard_normal(yt.shape))
    rx = np.concatenate([yt[..., N - C:], yt], axis=-1) if C > 0 else yt
    return {"rx": np.ascontiguousarray(rx.astype(np.complex64)), "pilot_asc": pilot_asc,
            "src_idx": src_idx, "h_true": h}


def make_frames_torch(n_frames, cfg, device, seed=None, snr_db="cfg", chunk=64):
    """Full-size batch built directly on `device` with torch (generator only; the receive
    path never uses torch.fft).  Returns (rx [F,S,A,N+C] complex64, pilot_asc numpy [K],
    src_idx [F,S-1,K] uint8 tensor in ascending-frequency order)."""
    import torch

    A, N, C, S, b = cfg.n_ant, cfg.fft_size, cfg.cp_len, cfg.n_sym, cfg.qam_bits
    K = N - 1
    seed = cfg.seed if seed is None else seed
    snr = cfg.snr_db if snr_db == "cfg" else snr_db
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    pilot_asc = make_pilot(K, seed)
    pil_bin = torch.from_numpy(asc_to_bin(pilot_asc)).to(device)
    lut = torch.from_numpy(qam_map_indices(np.arange(1 << b), b).astype(np.complex64)).to(device)
    rx = torch.empty((n_frames, S, A, N + C), dtype=torch.complex64, device=device)
    src = torch.empty((n_frames, S - 1, K), dtype=torch.uint8, device=device)
    shift = (K + 1) // 2
    for f0 in range(0, n_frames, chunk):
        nf = min(chunk, n_frames - f0)
        idx = torch.randint(0, 1 << b, (nf, S - 1, K), generator=g, device=device, dtype=torch.uint8)
        src[f0:f0 + nf] = idx
        tx = torch.zeros((nf, S, N), dtype=torch.complex64, device=device)
        tx[:, 0, 1:] = pil_bin
        tx[:, 1:, 1:] = torch.roll(lut[idx.long()], -shift, dims=-1)
        h = torch.zeros((nf, A, N), dtype=torch.complex64, device=device)
        hr = torch.randn((nf, A, K, 2), generator=g, device=device) * (0.5 ** 0.5)
        h[:, :, 1:] = torch.view_as_complex(hr)
        yt = torch.fft.ifft(tx[:, :, None, :] * h[:, None, :, :], dim=-1)
        if snr is not None:
            sigma = (K / (N * N) / (10.0 ** (snr / 10.0)) / 2.0) ** 0.5
            yt = yt + sigma * torch.view_as_complex(torch.randn((*yt.shape, 2), generator=g, device=device))
        rx[f0:f0 + nf, :, :, C:] = yt
        if C > 0:
            rx[f0:f0 + nf, :, :, :C] = yt[..., N - C:]
        del tx, h, hr, yt, idx
    return rx, pilot_asc, src


def _pilot_rows(pilot_asc, U, pilots):
    """(number of pilot symbols P, per-user pilot rows [U, K] ascending frequency) of a multi-user frame: time
    pilots, P = U (row u is the whole pilot, sent on symbol u), or comb pilots, P = 1 (row u is the pilot on the
    indices i = u mod U and zero elsewhere, all sent on symbol 0)"""
    K = pilot_asc.shape[0]
    rows = np.broadcast_to(pilot_asc.astype(np.complex128), (U, K)).copy()
    if pilots == "time":
        return U, rows
    if pilots != "comb":
        raise ValueError("pilots must be 'time' or 'comb'")
    rows[np.arange(K)[None, :] % U != np.arange(U)[:, None]] = 0.0
    return 1, rows


def make_frames_mu(n_frames, n_ant, fft_size, cp_len, n_sym, qam_bits, n_users, snr_db=None, seed=0, h=None, pilot_asc=None,
                   pilots="time"):
    """Multi-user uplink frames (include/ofdm_lsmrc.h, lsmrc_demod_frames_device_mu).  pilots="time": symbol u < U
    carries user u's pilot (the handle's pilot, the other users silent), symbols U..S-1 the data of all U users at once.
    pilots="comb": symbol 0 carries user u's pilot on the ascending-frequency indices i = u mod U (nothing elsewhere),
    symbols 1..S-1 the data.  i.i.d. Rayleigh channel per user, antenna and subcarrier; AWGN at `snr_db` per user and
    antenna.  `h` [F,U,A,K] (bin order, e.g. multipath_channel) replaces the random channel.  With n_users=1 and time
    pilots the random draws, their order and the arithmetic are those of make_frames: rx is byte-identical.  Returns
    dict(rx [F,S,A,N+C] c64, pilot_asc [K] c64, src_idx [F,S-P,U,K] u8 (ascending frequency; P = U time, 1 comb),
    h_true [F,U,A,K] c128 (bin order))."""
    F, A, N, C, S, U = n_frames, n_ant, fft_size, cp_len, n_sym, n_users
    K = N - 1
    rng = np.random.default_rng(seed)
    pilot_asc = make_pilot(K, seed) if pilot_asc is None else np.asarray(pilot_asc, np.complex64)
    P, prow = _pilot_rows(pilot_asc, U, pilots)
    assert 1 <= U and P < S
    src_idx = rng.integers(0, 1 << qam_bits, size=(F, S - P, U, K), dtype=np.uint8)
    data_asc = qam_map_indices(src_idx, qam_bits)
    tx_bin = np.zeros((F, S, U, N), np.complex128)
    for u in range(U):
        tx_bin[:, u if P == U else 0, u, 1:] = asc_to_bin(prow[u])
    tx_bin[:, P:, :, 1:] = asc_to_bin(data_asc)
    if h is None:
        h = (rng.standard_normal((F, U, A, K)) + 1j * rng.standard_normal((F, U, A, K))) / np.sqrt(2.0)
    else:
        h = np.asarray(h, np.complex128)
        assert h.shape == (F, U, A, K)
    hfull = np.zeros((F, U, A, N), np.complex128)
    hfull[..., 1:] = h
    yf = tx_bin[:, :, 0, None, :] * hfull[:, None, 0, :, :]    # [F,S,A,N]
    for u in range(1, U):
        yf = yf + tx_bin[:, :, u, None, :] * hfull[:, None, u, :, :]
    yt = np.fft.ifft(yf, axis=-1)
    if snr_db is not None:
        sig_pow = K / (N * N)
        sigma = np.sqrt(sig_pow / (10.0 ** (snr_db / 10.0)) / 2.0)
        yt = yt + sigma * (rng.standard_normal(yt.shape) + 1j * rng.standard_normal(yt.shape))
    rx = np.concatenate([yt[..., N - C:], yt], axis=-1) if C > 0 else yt
    return {"rx": np.ascontiguousarray(rx.astype(np.complex64)), "pilot_asc": pilot_asc,
            "src_idx": src_idx, "h_true": h}


def make_frames_mu_torch(n_frames, n_ant, fft_size, cp_len, n_sym, qam_bits, n_users, device, seed=0, snr_db=30.0,
                         chunk=16, pilots="time"):
    """make_frames_mu built directly on `device` with torch, for full-size batches (same frame formats, its own random
    stream).  Returns (rx [F,S,A,N+C] complex64 tensor, pilot_asc numpy [K], src_idx [F,S-P,U,K] uint8 tensor; P = U
    with time pilots, 1 with comb pilots)."""
    import torch

    A, N, C, S, U, b = n_ant, fft_size, cp_len, n_sym, n_users, qam_bits
    K = N - 1
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    pilot_asc = make_pilot(K, seed)
    P, prow = _pilot_rows(pilot_asc, U, pilots)
    assert 1 <= U and P < S
    pil_bin = torch.from_numpy(asc_to_bin(prow).astype(np.complex64)).to(device)   # [U,K]
    lut = torch.from_numpy(qam_map_indices(np.arange(1 << b), b).astype(np.complex64)).to(device)
    rx = torch.empty((n_frames, S, A, N + C), dtype=torch.complex64, device=device)
    src = torch.empty((n_frames, S - P, U, K), dtype=torch.uint8, device=device)
    shift = (K + 1) // 2
    for f0 in range(0, n_frames, chunk):
        nf = min(chunk, n_frames - f0)
        idx = torch.randint(0, 1 << b, (nf, S - P, U, K), generator=g, device=device, dtype=torch.uint8)
        src[f0:f0 + nf] = idx
        tx = torch.zeros((nf, S, U, N), dtype=torch.complex64, device=device)
        for u in range(U):
            tx[:, u if P == U else 0, u, 1:] = pil_bin[u]
        tx[:, P:, :, 1:] = torch.roll(lut[idx.long()], -shift, dims=-1)
        h = torch.zeros((nf, U, A, N), dtype=torch.complex64, device=device)
        h[..., 1:] = torch.view_as_complex(torch.randn((nf, U, A, K, 2), generator=g, device=device) * (0.5 ** 0.5))
        yf = torch.einsum("fsun,fuan->fsan", tx, h)
        yt = torch.fft.ifft(yf, dim=-1)
        if snr_db is not None:
            sigma = (K / (N * N) / (10.0 ** (snr_db / 10.0)) / 2.0) ** 0.5
            yt = yt + sigma * torch.view_as_complex(torch.randn((*yt.shape, 2), generator=g, device=device))
        rx[f0:f0 + nf, :, :, C:] = yt
        if C > 0:
            rx[f0:f0 + nf, :, :, :C] = yt[..., N - C:]
        del tx, h, yf, yt, idx
    return rx, pilot_asc, src


def multipath_channel(n_frames, n_users, n_ant, fft_size, n_taps, seed=0):
    """Frequency response of a tapped delay line per (frame, user, antenna): n_taps independent complex Gaussian taps at
    the integer delays 0 .. n_taps-1, each of power 1 / n_taps (E|H|^2 = 1).  H[bin] = sum_l g_l exp(-2 pi j bin l / N)
    on bins 1..N-1.  Unlike the i.i.d. Rayleigh draw of make_frames_mu it is smooth in frequency, so comb pilots can be
    interpolated.  Returns [F,U,A,K] complex128, bin order (make_frames_mu's `h`)."""
    rng = np.random.default_rng(seed)
    shape = (n_frames, n_users, n_ant, n_taps)
    g = (rng.standard_normal(shape) + 1j * rng.standard_normal(shape)) / np.sqrt(2.0 * n_taps)
    ph = np.exp(-2j * np.pi * np.outer(np.arange(n_taps), np.arange(1, fft_size)) / fft_size)   # [L,K]
    return g @ ph


def make_pn(length=255, seed=0x1D):
    """+-1 maximal-length sequence (8-bit LFSR x^8+x^6+x^5+x^4+1 -> period 255), as complex64.  Stands in for
    the reference's PNSeq_255_MaxLenSeq.dat (rx_and_corr.cpp:228), which is not shipped."""
    reg = seed & 0xFF or 1
    out = np.empty(length, np.float32)
    for i in range(length):
        out[i] = 1.0 if (reg & 1) else -1.0
        fb = ((reg >> 0) ^ (reg >> 2) ^ (reg >> 3) ^ (reg >> 4)) & 1
        reg = (reg >> 1) | (fb << 7)
    return out.astype(np.complex64)


def make_capture(rx_frame, pn, offset, samps=None, noise=0.02, seed=0):
    """Wrap one frame [S][A][N+C] into the two per-channel capture buffers the reference's receive loop sees
    (rx_and_corr.cpp:305-312): noise, then conj(pn) starting at `offset` of buffer 1 (the correlator multiplies by
    pn without conjugating, :348), then the frame, whose tail wraps into buffer 2.  Returns (buf1, buf2) [A][samps]."""
    S, A, row = rx_frame.shape
    L = pn.shape[0]
    frame = np.ascontiguousarray(np.transpose(rx_frame, (1, 0, 2))).reshape(A, S * row)   # [A][S*row]
    samps = samps or (L + S * row)
    assert samps - L >= S * row and 0 <= offset and offset + L <= samps
    rng = np.random.default_rng(seed)
    scale = float(np.abs(frame).mean()) or 1.0
    def noise_buf():
        return (noise * scale * (rng.standard_normal((A, samps)) + 1j * rng.standard_normal((A, samps)))).astype(np.complex64)
    buf1, buf2 = noise_buf(), noise_buf()
    buf1[:, offset:offset + L] = np.conj(pn)[None, :]
    n_first = samps - offset - L
    stream = np.concatenate([frame, noise_buf()[:, :max(0, samps - L - S * row)]], axis=1)  # samps-L per channel
    buf1[:, offset + L:] = stream[:, :n_first]
    buf2[:, :offset] = stream[:, n_first:n_first + offset]
    return buf1, buf2
