"""ctypes binding of include/ofdm_lsmrc.h -- the same C ABI any other host language
would bind (see INTEGRATION.md).  No compute happens in Python: every method is one
call into libofdm_lsmrc.so, which launches the sm_100a kernels.  There is no CPU
fallback; a missing library or a missing GPU raises.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, byref, c_char_p, c_float, c_int, c_longlong, c_size_t, c_void_p

import numpy as np

from . import build as _build

LSMRC_OK = 0
ERR_NAMES = {0: "LSMRC_OK", -1: "LSMRC_ERR_INVALID", -2: "LSMRC_ERR_CUDA", -3: "LSMRC_ERR_UNSUPPORTED",
             -4: "LSMRC_ERR_NO_PILOT", -5: "LSMRC_ERR_NO_DEVICE", -6: "LSMRC_ERR_STATE"}

# every symbol include/ofdm_lsmrc.h declares: name -> (restype, argtypes)
ABI = {
    "lsmrc_abi_version": (c_int, []),
    "lsmrc_create": (c_int, [c_void_p, POINTER(c_void_p)]),
    "lsmrc_destroy": (c_int, [c_void_p]),
    "lsmrc_last_error": (c_char_p, [c_void_p]),
    "lsmrc_error_name": (c_char_p, [c_int]),
    "lsmrc_bits_row_bytes": (c_size_t, [c_int, c_int]),
    "lsmrc_rx_frame_elems": (c_size_t, [c_void_p]),
    "lsmrc_supported_fft_size": (c_int, [c_int]),
    "lsmrc_set_pilot": (c_int, [c_void_p, c_void_p, c_int]),
    "lsmrc_set_pilot_file": (c_int, [c_void_p, c_char_p]),
    "lsmrc_demod_frames_device": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p]),
    "lsmrc_demod_frames_device_soft": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_float]),
    "lsmrc_demod_frames_host": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p]),
    "lsmrc_demod_frames_host_sc16": (c_int, [c_void_p, c_void_p, c_int, c_float, c_void_p, c_void_p, c_void_p, c_void_p]),
    "lsmrc_sc16_to_fc32_device": (c_int, [c_void_p, c_void_p, c_longlong, c_int, c_int, c_int, c_float, c_void_p]),
    "lsmrc_first_vector": (c_int, [c_void_p, c_void_p, c_int]),
    "lsmrc_demod_one_symbol": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_void_p]),
    "lsmrc_get_channel": (c_int, [c_void_p, c_void_p, c_void_p]),
    "lsmrc_get_channel_device": (c_int, [c_void_p, c_void_p, c_void_p]),
    "lsmrc_ring_submit_frame": (c_int, [c_void_p, c_int, c_void_p, c_size_t]),
    "lsmrc_ring_prepare": (c_int, [c_void_p]),
    "lsmrc_set_one_launch_frames": (c_int, [c_void_p, c_int]),
    "lsmrc_one_launch_frames_count": (c_longlong, [c_void_p]),
    "lsmrc_ring_submit_split": (c_int, [c_void_p, c_int, c_void_p, c_int, c_void_p]),
    "lsmrc_ring_wait": (c_int, [c_void_p, c_int, POINTER(c_void_p), POINTER(c_void_p), POINTER(c_void_p)]),
    "lsmrc_ring_copy_done": (c_int, [c_void_p, c_int]),
    "lsmrc_stage_drop_prefix": (c_int, [c_void_p, c_void_p, c_void_p, c_longlong]),
    "lsmrc_stage_fft": (c_int, [c_void_p, c_void_p, c_longlong]),
    "lsmrc_stage_find_hs": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p]),
    "lsmrc_stage_find_hsqrd": (c_int, [c_void_p, c_void_p, c_void_p]),
    "lsmrc_stage_mult_conj": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int]),
    "lsmrc_stage_combine": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int]),
    "lsmrc_stage_shift_rows": (c_int, [c_void_p, c_void_p, c_void_p, c_longlong]),
    "lsmrc_copy_device": (c_int, [c_void_p, c_void_p, c_void_p, c_size_t]),
    "lsmrc_sync_correlate": (c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p, c_int, c_float, POINTER(c_int), POINTER(c_int),
                                     POINTER(c_float), c_void_p]),
    "lsmrc_sync_assemble": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    "lsmrc_dev_alloc": (c_int, [c_void_p, c_size_t, POINTER(c_void_p)]),
    "lsmrc_dev_free": (c_int, [c_void_p, c_void_p]),
    "lsmrc_copy_to_device": (c_int, [c_void_p, c_void_p, c_void_p, c_size_t]),
    "lsmrc_copy_to_host": (c_int, [c_void_p, c_void_p, c_void_p, c_size_t]),
    "lsmrc_host_alloc": (c_int, [c_void_p, c_size_t, POINTER(c_void_p)]),
    "lsmrc_host_free": (c_int, [c_void_p, c_void_p]),
    "lsmrc_host_register": (c_int, [c_void_p, c_void_p, c_size_t]),
    "lsmrc_host_unregister": (c_int, [c_void_p, c_void_p]),
    "lsmrc_set_stream": (c_int, [c_void_p, c_void_p]),
    "lsmrc_ring_trace": (c_int, [c_void_p, c_int, c_void_p]),
    "lsmrc_device_count": (c_int, []),
    "lsmrc_device_pci_bus_id": (c_int, [c_int, c_char_p, c_size_t]),
    "lsmrc_sync": (c_int, [c_void_p]),
    "lsmrc_estimate_noise_var": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_void_p]),
    "lsmrc_llr_from_combined": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p]),
    "lsmrc_zf_create": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, POINTER(c_int)]),
    "lsmrc_zf_apply": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    "lsmrc_demod_frames_device_mu": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_float, c_void_p, c_void_p, c_void_p,
                                             POINTER(c_int)]),
    "lsmrc_demod_frames_device_mu_soft": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_float, c_void_p, c_void_p, c_void_p,
                                                  c_void_p, c_void_p, POINTER(c_int)]),
    "lsmrc_set_mu_pilots": (c_int, [c_void_p, c_int]),
    "lsmrc_precode_frames_device": (c_int, [c_void_p, c_void_p, c_int, c_int, c_float, c_void_p, c_int, c_void_p, c_void_p,
                                            POINTER(c_int)]),
    "lsmrc_ring_copy_query": (c_int, [c_void_p, c_int]),
    "lsmrc_ring_submit_frames": (c_int, [c_void_p, c_int, c_void_p, c_int, c_void_p, c_int]),
    "lsmrc_set_timing": (c_int, [c_void_p, c_int]),
    "lsmrc_set_oneshot": (c_int, [c_void_p, c_int]),
    "lsmrc_oneshot_count": (ctypes.c_longlong, [c_void_p]),
    "lsmrc_last_kernel_ms": (c_int, [c_void_p, POINTER(c_float), POINTER(c_float)]),
    "lsmrc_kernel_ms_history": (c_int, [c_void_p, c_int, POINTER(c_float), POINTER(c_float), POINTER(c_int)]),
    "lsmrc_launch_count": (c_longlong, [c_void_p]),
    "lsmrc_describe_plan": (c_int, [c_void_p, c_char_p, c_size_t]),
}


class LsmrcConfig(ctypes.Structure):
    _fields_ = [("n_ant", c_int), ("fft_size", c_int), ("cp_len", c_int), ("n_sym", c_int),
                ("qam_bits", c_int), ("max_frames", c_int), ("device", c_int), ("n_lanes", c_int)]


class LsmrcError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"{ERR_NAMES.get(code, code)}: {msg}")
        self.code = code


_LIB = None


def load_library(path: str | None = None) -> ctypes.CDLL:
    """Load libofdm_lsmrc.so (building it in-tree first if it is missing or stale)."""
    global _LIB
    if _LIB is not None and path is None:
        return _LIB
    path = path or os.environ.get("LSMRC_LIB") or None
    p = path or _build.LIB_PATH
    if path is None and _build.needs_build():
        _build.build()
    if not os.path.exists(p):
        raise RuntimeError(f"{p} is missing: the CUDA library is the product, there is no fallback")
    lib = ctypes.CDLL(p)
    for name, (res, args) in ABI.items():
        fn = getattr(lib, name)  # AttributeError if the library does not export it
        fn.restype = res
        fn.argtypes = args
    if lib.lsmrc_abi_version() != 1:
        raise RuntimeError("ABI version mismatch")
    if path is None:
        _LIB = lib
    return lib


def _ptr(x):
    """device/host pointer of a numpy array, torch tensor, int or None"""
    if x is None:
        return None
    if isinstance(x, int):
        return x
    if isinstance(x, np.ndarray):
        if not x.flags["C_CONTIGUOUS"]:
            raise ValueError("array must be C-contiguous")
        return x.ctypes.data
    if hasattr(x, "data_ptr"):
        if not x.is_contiguous():
            raise ValueError("tensor must be contiguous")
        return x.data_ptr()
    raise TypeError(type(x))


class LsMrcReceiver:
    """Host-side handle: one per (dimensions, device).  Mirrors the call sequence of
    gpuLS_main.cu:66-141 (create -> pilot -> firstVector/demodOneSymbol or whole frames)."""

    def __init__(self, n_ant, fft_size, cp_len, n_sym, qam_bits, max_frames=1, device=0, n_lanes=3):
        self.lib = load_library()
        self.cfg = LsmrcConfig(n_ant, fft_size, cp_len, n_sym, qam_bits, max_frames, device, n_lanes)
        self.K = fft_size - 1
        self.row_bytes = (self.K * qam_bits + 7) // 8
        h = c_void_p()
        rc = self.lib.lsmrc_create(byref(self.cfg), byref(h))
        if rc != LSMRC_OK:
            raise LsmrcError(rc, (self.lib.lsmrc_last_error(None) or b"").decode())
        self.h = h

    @classmethod
    def from_config(cls, cfg, **kw):
        return cls(cfg.n_ant, cfg.fft_size, cfg.cp_len, cfg.n_sym, cfg.qam_bits, **kw)

    def _ck(self, rc):
        if rc < 0:
            raise LsmrcError(rc, (self.lib.lsmrc_last_error(self.h) or b"").decode())
        return rc

    def close(self):
        if getattr(self, "h", None):
            for p in getattr(self, "_pinned", []):  # buffers handed out by pinned_array()
                self.lib.lsmrc_host_free(self.h, p)
            self._pinned = []
            self.lib.lsmrc_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    # -- pilot
    def set_pilot(self, pilot_asc):
        p = np.ascontiguousarray(pilot_asc, dtype=np.complex64)
        self._ck(self.lib.lsmrc_set_pilot(self.h, p.ctypes.data, p.shape[0]))

    def set_pilot_file(self, path):
        return self._ck(self.lib.lsmrc_set_pilot_file(self.h, path.encode() if path else None))

    # -- whole frames
    def demod_frames_device(self, d_rx, n_frames, d_combined, d_bits=None, d_hconj=None, d_hsqrd=None):
        self._ck(self.lib.lsmrc_demod_frames_device(self.h, _ptr(d_rx), n_frames, _ptr(d_hconj), _ptr(d_hsqrd),
                                                    _ptr(d_combined), _ptr(d_bits)))

    def demod_frames_device_soft(self, d_rx, n_frames, d_combined, d_llr, noise_var, d_bits=None):
        self._ck(self.lib.lsmrc_demod_frames_device_soft(self.h, _ptr(d_rx), n_frames, _ptr(d_combined), _ptr(d_bits),
                                                         _ptr(d_llr), noise_var))

    def estimate_noise_var(self, d_combined, d_hsqrd, n_frames, d_noise_var):
        self._ck(self.lib.lsmrc_estimate_noise_var(self.h, _ptr(d_combined), _ptr(d_hsqrd), n_frames, _ptr(d_noise_var)))

    def llr_from_combined(self, d_combined, d_hsqrd, d_noise_var, n_frames, d_llr):
        self._ck(self.lib.lsmrc_llr_from_combined(self.h, _ptr(d_combined), _ptr(d_hsqrd), _ptr(d_noise_var), n_frames, _ptr(d_llr)))

    def zf_create(self, d_x, n_ant, n_sc, n_users, d_hzf) -> int:
        """multi-user zero-forcing matrices (cpuLS.hpp:415-447); returns the number of singular subcarriers"""
        bad = c_int()
        self._ck(self.lib.lsmrc_zf_create(self.h, _ptr(d_x), n_ant, n_sc, n_users, _ptr(d_hzf), byref(bad)))
        return bad.value

    DETECTORS = {"zf": 0, "mmse": 1}
    MU_PILOTS = {"time": 0, "comb": 1}

    def set_mu_pilots(self, layout="time"):
        """Pilot layout of the multi-user calls on this handle: "time" (default; symbols 0..U-1 carry one user's pilot
        each) or "comb" (symbol 0 carries every user's pilot, user u on the ascending-frequency indices i = u mod U;
        each user's channel is interpolated across its own subcarriers).  Read when a call is enqueued."""
        self._ck(self.lib.lsmrc_set_mu_pilots(self.h, self.MU_PILOTS.get(layout, -1)))

    def demod_frames_device_mu(self, d_rx, n_frames, n_users, d_combined, d_bits=None, d_hconj=None, detector="zf",
                               noise_var=0.0, count_singular=False):
        """Multi-user frames: P pilot symbols, then symbols P..S-1 with the data of all users; per-user LS channel and ZF
        or MMSE detection.  Time pilots (P = U): d_combined [F,S-U,U,K], d_bits [F,S-U,U,row].  Comb pilots (P = 1,
        set_mu_pilots("comb")): d_combined [F,S-1,U,K], d_bits [F,S-1,U,row].  d_hconj [F,U,A,K] in both.  With
        count_singular the call is synchronous and returns the number of (frame, subcarrier) pairs whose Gram matrix
        was singular."""
        bad = c_int(0)
        self._ck(self.lib.lsmrc_demod_frames_device_mu(self.h, _ptr(d_rx), n_frames, n_users, self.DETECTORS.get(detector, -1),
                                                       float(noise_var), _ptr(d_hconj), _ptr(d_combined), _ptr(d_bits),
                                                       byref(bad) if count_singular else None))
        return bad.value if count_singular else None

    def demod_frames_device_mu_soft(self, d_rx, n_frames, n_users, d_combined, d_llr, d_bits=None, d_hconj=None, d_sinr=None,
                                    detector="zf", noise_var=1.0, count_singular=False):
        """demod_frames_device_mu plus soft output: d_llr float32 max-log LLRs (LLR > 0 <=> bit 0), [F,S-U,U,K,b] with
        time pilots and [F,S-1,U,K,b] with comb pilots, and d_sinr [F,U,K] float32 post-detection SINR, both ascending
        frequency.  noise_var (> 0, both detectors) is the
        noise variance per antenna and subcarrier; MMSE uses it as its diagonal loading too.  d_combined and d_bits are
        those of demod_frames_device_mu (for MMSE the biased estimate; the LLRs use the unbiased one)."""
        bad = c_int(0)
        self._ck(self.lib.lsmrc_demod_frames_device_mu_soft(self.h, _ptr(d_rx), n_frames, n_users, self.DETECTORS.get(detector, -1),
                                                            float(noise_var), _ptr(d_hconj), _ptr(d_combined), _ptr(d_bits),
                                                            _ptr(d_llr), _ptr(d_sinr), byref(bad) if count_singular else None))
        return bad.value if count_singular else None

    def precode_frames_device(self, d_hconj, n_frames, n_users, d_sym, n_sym_dl, d_tx, d_gain=None, reg=0.0,
                              count_singular=False):
        """Multi-user downlink: ZF (reg = 0) or regularised-ZF precoding from the uplink estimate d_hconj [F,U,A,K] (as
        demod_frames_device_mu exports it), inverse FFT and cyclic prefix.  d_sym [F,Sd,U,K] complex64 ascending
        frequency -> d_tx [F,Sd,A,N+C] complex64, d_gain [F] float32 per-frame power gain.  With count_singular the call
        is synchronous and returns the number of (frame, subcarrier) pairs whose Gram matrix was singular."""
        bad = c_int(0)
        self._ck(self.lib.lsmrc_precode_frames_device(self.h, _ptr(d_hconj), n_frames, n_users, float(reg), _ptr(d_sym), n_sym_dl,
                                                      _ptr(d_tx), _ptr(d_gain), byref(bad) if count_singular else None))
        return bad.value if count_singular else None

    def zf_apply(self, d_hzf, d_xd, n_ant, n_sc, n_users, d_hx):
        self._ck(self.lib.lsmrc_zf_apply(self.h, _ptr(d_hzf), _ptr(d_xd), n_ant, n_sc, n_users, _ptr(d_hx)))

    def demod_frames_host(self, h_rx, n_frames, h_combined, h_bits=None, h_hconj=None, h_hsqrd=None):
        self._ck(self.lib.lsmrc_demod_frames_host(self.h, _ptr(h_rx), n_frames, _ptr(h_hconj), _ptr(h_hsqrd),
                                                  _ptr(h_combined), _ptr(h_bits)))

    def set_one_launch_frames(self, enabled: bool):
        self._ck(self.lib.lsmrc_set_one_launch_frames(self.h, int(enabled)))

    def one_launch_frames_count(self) -> int:
        return int(self.lib.lsmrc_one_launch_frames_count(self.h))

    def demod_frames_host_sc16(self, h_rx_iq, n_frames, scale, h_combined, h_bits=None, h_hconj=None, h_hsqrd=None):
        """frames in the radio's wire format: h_rx_iq [F,S,A,N+C,2] int16, sample = int16 * scale (converted on the device)"""
        self._ck(self.lib.lsmrc_demod_frames_host_sc16(self.h, _ptr(h_rx_iq), n_frames, float(scale), _ptr(h_hconj), _ptr(h_hsqrd),
                                                       _ptr(h_combined), _ptr(h_bits)))

    def sc16_to_fc32_device(self, d_iq, rows, row_len_in, skip, row_len_out, scale, d_out):
        self._ck(self.lib.lsmrc_sc16_to_fc32_device(self.h, _ptr(d_iq), rows, row_len_in, skip, row_len_out, float(scale), _ptr(d_out)))

    def demod_numpy(self, rx: np.ndarray, want_channel=True):
        """Convenience for tests: rx [F,S,A,N+C] complex64 host array -> dict of host arrays."""
        rx = np.ascontiguousarray(rx, dtype=np.complex64)
        F, S, A, NC = rx.shape
        c = self.cfg
        assert (S, A, NC) == (c.n_sym, c.n_ant, c.fft_size + c.cp_len), "shape does not match the handle"
        comb = np.empty((F, S - 1, self.K), np.complex64)
        bits = np.empty((F, S - 1, self.row_bytes), np.uint8)
        hc = np.empty((F, A, self.K), np.complex64) if want_channel else None
        hs = np.empty((F, self.K), np.float32) if want_channel else None
        self.demod_frames_host(rx, F, comb, bits, hc, hs)
        return {"combined": comb, "bits": bits, "hconj": hc, "hsqrd": hs}

    # -- per symbol (firstVector / demodOneSymbol)
    def first_vector(self, rx_sym, on_device=False):
        self._ck(self.lib.lsmrc_first_vector(self.h, _ptr(rx_sym), int(on_device)))

    def demod_one_symbol(self, rx_sym, on_device=False):
        comb = np.empty(self.K, np.complex64)
        bits = np.empty(self.row_bytes, np.uint8)
        self._ck(self.lib.lsmrc_demod_one_symbol(self.h, _ptr(rx_sym), int(on_device), comb.ctypes.data, bits.ctypes.data))
        return comb, bits

    def get_channel(self):
        hc = np.empty((self.cfg.n_ant, self.K), np.complex64)
        hs = np.empty(self.K, np.float32)
        self._ck(self.lib.lsmrc_get_channel(self.h, hc.ctypes.data, hs.ctypes.data))
        return hc, hs

    # -- ring lanes
    def ring_submit_frame(self, lane, h_slots, slot_stride_bytes=None):
        stride = slot_stride_bytes or 8 * self.cfg.n_ant * (self.cfg.fft_size + self.cfg.cp_len)
        self._ck(self.lib.lsmrc_ring_submit_frame(self.h, lane, _ptr(h_slots), stride))

    def ring_wait(self, lane):
        c, b, hc = c_void_p(), c_void_p(), c_void_p()
        self._ck(self.lib.lsmrc_ring_wait(self.h, lane, byref(c), byref(b), byref(hc)))
        nd = self.cfg.n_sym - 1
        comb = np.ctypeslib.as_array(ctypes.cast(c, POINTER(c_float)), shape=(nd, self.K, 2)).view(np.complex64)[..., 0]
        bits = np.ctypeslib.as_array(ctypes.cast(b, POINTER(ctypes.c_uint8)), shape=(nd, self.row_bytes))
        return comb, bits

    # -- stand-alone steps (device pointers / torch tensors)
    def stage(self, name, *args):
        fn = getattr(self.lib, "lsmrc_stage_" + name)
        self._ck(fn(self.h, *[_ptr(a) for a in args]))

    # -- receive front end (device tensors)
    def sync_correlate(self, d_buf, n_chan, samps, d_pn, pn_len, thres, d_metric_all=None):
        off, ch, m = c_int(), c_int(), c_float()
        self._ck(self.lib.lsmrc_sync_correlate(self.h, _ptr(d_buf), n_chan, samps, _ptr(d_pn), pn_len, thres, byref(off),
                                               byref(ch), byref(m), _ptr(d_metric_all)))
        return off.value, ch.value, m.value

    def sync_assemble(self, d_buf1, d_buf2, samps, offset, pn_len, d_rx_frame):
        self._ck(self.lib.lsmrc_sync_assemble(self.h, _ptr(d_buf1), _ptr(d_buf2), samps, offset, pn_len, _ptr(d_rx_frame)))

    # -- plumbing
    def host_alloc(self, nbytes):
        p = c_void_p()
        self._ck(self.lib.lsmrc_host_alloc(self.h, nbytes, byref(p)))
        return p.value

    def host_free(self, p):
        self._ck(self.lib.lsmrc_host_free(self.h, p))

    def host_register(self, arr):
        self._ck(self.lib.lsmrc_host_register(self.h, _ptr(arr), arr.nbytes))

    def host_unregister(self, arr):
        self._ck(self.lib.lsmrc_host_unregister(self.h, _ptr(arr)))

    def pinned_array(self, shape, dtype):
        """numpy array backed by pinned host memory owned by this handle: freed by close(), after which the
        array must not be touched."""
        n = int(np.prod(shape)) * np.dtype(dtype).itemsize
        p = self.host_alloc(max(n, 1))
        if not hasattr(self, "_pinned"):
            self._pinned = []
        self._pinned.append(p)
        buf = (ctypes.c_char * max(n, 1)).from_address(p)
        return np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)

    def set_stream(self, stream_ptr):
        self._ck(self.lib.lsmrc_set_stream(self.h, stream_ptr))

    def sync(self):
        self._ck(self.lib.lsmrc_sync(self.h))

    def set_oneshot(self, mode=2):
        """Launch policy for launch-latency-bound batches: 2 (default) one fused kernel, pinned host buffers
        processed in place; 1 fused kernel with staged copies; 0 always pilot + data kernels."""
        self._ck(self.lib.lsmrc_set_oneshot(self.h, int(mode)))

    def oneshot_count(self) -> int:
        return int(self.lib.lsmrc_oneshot_count(self.h))

    def set_timing(self, on=True):
        self._ck(self.lib.lsmrc_set_timing(self.h, int(on)))

    def last_kernel_ms(self):
        a, b = c_float(), c_float()
        self._ck(self.lib.lsmrc_last_kernel_ms(self.h, byref(a), byref(b)))
        return a.value, b.value

    def kernel_ms_history(self, max_n=256):
        a = (c_float * max_n)()
        b = (c_float * max_n)()
        n = c_int()
        self._ck(self.lib.lsmrc_kernel_ms_history(self.h, max_n, a, b, byref(n)))
        return list(a[:n.value]), list(b[:n.value])

    def launch_count(self):
        return int(self.lib.lsmrc_launch_count(self.h))

    def describe_plan(self):
        buf = ctypes.create_string_buffer(256)
        self._ck(self.lib.lsmrc_describe_plan(self.h, buf, 256))
        return buf.value.decode()
