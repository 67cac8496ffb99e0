/*
 * ofdm_lsmrc.h -- C ABI of the B200-native uplink OFDM receiver hot path
 * (CP strip -> per-antenna FFT -> LS channel estimate -> MRC -> hard QAM demap).
 *
 * This is the drop-in boundary for the reference's GPU path: the reference has no
 * FFI layer, its surface is `class gpuLS` (gpuLS.cuh:72-113) driven by
 * gpuLS_main.cu:66-141 plus the ShMemSymBuff ring.  Every entry point below names
 * the reference interface it replaces.  Plain pointers and sizes only; no CUDA,
 * torch or C++ types cross this boundary, so the C++ facade in
 * gpu-accel-ofdm-ls-mrc_b200/host/ (same class and method names as the reference)
 * and any other binding (ctypes, cgo, JNI ...) can sit on top of it.
 *
 * Dimensions are runtime here; the reference fixes them with -D macros
 * (ShMemSymBuff.hpp:42-67): A = numOfRows, N = dimension, C = prefix,
 * S = lenOfBuffer (symbol 0 of a frame is the pilot), K = N-1 used subcarriers.
 *
 * Data layouts (all complex64 = interleaved float re,im -- complexF /
 * cuFloatComplex, ShMemSymBuff.hpp:86-89):
 *   rx        [F][S][A][N+C]  antenna-samples exactly as the ring slots hold them
 *                             (struct symbol, ShMemSymBuff.hpp:92-94), CP included
 *   pilot     [K]             ascending frequency, the Pilots.dat order (cpuLS.hpp:93)
 *   hconj     [F][A][K]       conj(H), FFT-bin order (bin k+1 at index k) -- what the
 *                             reference keeps in dH/Hconj (gpuLS.cu:158-182)
 *   hsqrd     [F][K]          sum_a |H|^2 (float)      (gpuLS.cu:185-209)
 *   combined  [F][S-1][K]     MRC output, ascending frequency -- the Output_gpu.dat
 *                             record order (gpuLS_main.cu:114-126)
 *   bits      [F][S-1][row]   hard-demapped bits, LSB first, symbol i at stream bits
 *                             [i*b, i*b+b) of its row; row = lsmrc_bits_row_bytes()
 *
 * There is no CPU fallback: every compute entry point fails with
 * LSMRC_ERR_NO_DEVICE / LSMRC_ERR_CUDA when no sm_100 GPU is usable.
 * Error convention: 0 on success, negative LSMRC_ERR_* otherwise (the reference
 * ignores every CUDA status and returns void); lsmrc_last_error() gives text.
 */
#ifndef OFDM_LSMRC_H
#define OFDM_LSMRC_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LSMRC_ABI_VERSION 1

enum {
    LSMRC_OK = 0,
    LSMRC_ERR_INVALID = -1,     /* bad argument / dimension */
    LSMRC_ERR_CUDA = -2,        /* a CUDA runtime call failed */
    LSMRC_ERR_UNSUPPORTED = -3, /* FFT size or QAM order not built */
    LSMRC_ERR_NO_PILOT = -4,    /* lsmrc_set_pilot* not called yet */
    LSMRC_ERR_NO_DEVICE = -5,   /* no CUDA device / not sm_100 */
    LSMRC_ERR_STATE = -6        /* call order (e.g. data symbol before pilot symbol) */
};

typedef struct lsmrc_ctx *lsmrc_handle;

typedef struct lsmrc_config {
    int n_ant;      /* A: numOfRows   (ShMemSymBuff.hpp:42-44) */
    int fft_size;   /* N: dimension   (ShMemSymBuff.hpp:46-48), power of two 64..4096 */
    int cp_len;     /* C: prefix      (ShMemSymBuff.hpp:50-52) */
    int n_sym;      /* S: lenOfBuffer (ShMemSymBuff.hpp:63-65), pilot + S-1 data symbols */
    int qam_bits;   /* 2 (QPSK), 4 (16-QAM), 6 (64-QAM) */
    int max_frames; /* frames per chunk of the host-buffer path (device staging capacity) */
    int device;     /* CUDA ordinal; the reference hard-codes 0 (gpuLS_main.cu:69) */
    int n_lanes;    /* copy/compute lanes (streams) of the host-buffer and ring paths, >= 1 */
} lsmrc_config;

/* ---- lifetime (replaces gpuLS::gpuLS(), gpuLS.cu:43-47, and the cudaMalloc block of
 *      gpuLS_main.cu:73-91) ------------------------------------------------------- */
int lsmrc_abi_version(void);
int lsmrc_create(const lsmrc_config *cfg, lsmrc_handle *out);
int lsmrc_destroy(lsmrc_handle h);
const char *lsmrc_last_error(lsmrc_handle h); /* h may be NULL: last create() failure */
const char *lsmrc_error_name(int code);

/* ---- geometry helpers -------------------------------------------------------------- */
size_t lsmrc_bits_row_bytes(int fft_size, int qam_bits);         /* ceil((N-1)*b/8) */
size_t lsmrc_rx_frame_elems(const lsmrc_config *cfg);            /* S*A*(N+C) complex */
int lsmrc_supported_fft_size(int fft_size);
/* multi-GPU hosts (one handle and one worker thread per GPU; gpuLS_main.cu:69 pins the reference to device 0):
 * number of CUDA devices, and "dddd:bb:dd.f" of one of them (to find its NUMA node under /sys/bus/pci/devices) */
int lsmrc_device_count(void);
int lsmrc_device_pci_bus_id(int device, char *buf, size_t buf_len);                      /* 1 if a plan is built */

/* ---- pilot (replaces gpuLS::matrix_readX, gpuLS.cu:53-86, and copyPilotToGPU :88-106) - */
/* pilot_asc: K complex64 in ascending-frequency (file) order; rolled to bin order inside. */
int lsmrc_set_pilot(lsmrc_handle h, const float *pilot_asc, int K);
/* Reads K complex64 from `path` (Pilots.dat format).  When the file cannot be opened the
 * CPU reference's fallback 0.707+0.707i is used (cpuLS.hpp:85-88) and 1 is returned. */
int lsmrc_set_pilot_file(lsmrc_handle h, const char *path);

/* ---- whole frames, device-resident (replaces gpuLS::demodOneFrameCUDA gpuLS.cu:575 /
 *      demodOptimized :677 / demodCuBlas :771).  All pointers are DEVICE pointers.
 *      d_hconj / d_hsqrd / d_bits may be NULL (internal scratch / skipped).  The work is
 *      enqueued on the handle's compute stream; call lsmrc_sync() before reading.  That
 *      stream is the handle's own NON-BLOCKING stream unless lsmrc_set_stream was called: it
 *      does not order against the legacy default stream, so work the caller still has in flight
 *      on the buffers elsewhere (a fill of the outputs, the upload of d_rx) must have finished,
 *      or the caller passes its own stream with lsmrc_set_stream and enqueues everything there.
 *      On the caller's stream a call can also be captured into a CUDA graph and replayed (after one
 *      ordinary call of the same size, which allocates the per-frame channel state): the kernels
 *      keep their work counters on the device and re-arm them themselves, nothing is mirrored on
 *      the host (tests/test_gpu_parity.py::test_device_calls_replay_from_a_cuda_graph). */
int lsmrc_demod_frames_device(lsmrc_handle h, const void *d_rx, int n_frames, void *d_hconj,
                              void *d_hsqrd, void *d_combined, void *d_bits);

/* Same as lsmrc_demod_frames_device plus soft output (SURVEY 8f, rank 2 -- not in the reference):
 * d_llr [F][S-1][K][b] float, ascending frequency, bit order as in the packed bits, LLR > 0 <=> bit 0.
 * Max-log piecewise-linear LLRs scaled by the post-MRC SNR sum|H|^2 / noise_var (noise_var: noise variance
 * per antenna and subcarrier after the FFT, supplied by the caller).  d_bits may be NULL.
 * noise_var must be finite and > 0 with a finite float reciprocal (>= 1/FLT_MAX, about 2.9e-39): anything else
 * (0, negative, NaN, +inf, smaller subnormals) is LSMRC_ERR_INVALID and nothing is launched. */
int lsmrc_demod_frames_device_soft(lsmrc_handle h, const void *d_rx, int n_frames, void *d_combined,
                                   void *d_bits, void *d_llr, float noise_var);

/* Noise variance when the caller does not know it (SURVEY 8f rank 2, second half -- not in the reference):
 * decision-directed estimate per frame from the receiver's own outputs,
 *   noise_var[f] = mean over data symbols s, subcarriers i of  sum|H|^2[f][bin(i)] * |y[f][s][i] - slice(y[f][s][i])|^2
 * (after MRC the symbol error has variance noise_var / sum|H|^2; slice = nearest constellation point).
 * d_combined [F][S-1][K] and d_hsqrd [F][K] as written by lsmrc_demod_frames_device; d_noise_var [F] float.
 * lsmrc_llr_from_combined then turns the combined symbols into the same max-log LLRs as
 * lsmrc_demod_frames_device_soft, scaled per frame by d_noise_var[f] (d_llr [F][S-1][K][b]).
 * Both touch only the outputs (1/A of the input bytes); deterministic reduction order. */
int lsmrc_estimate_noise_var(lsmrc_handle h, const void *d_combined, const void *d_hsqrd, int n_frames, void *d_noise_var);
int lsmrc_llr_from_combined(lsmrc_handle h, const void *d_combined, const void *d_hsqrd, const void *d_noise_var, int n_frames,
                            void *d_llr);

/* ---- whole frames, host buffers (replaces gpuLS::demodOneFrame gpuLS.cu:475: H2D,
 *      compute, D2H inside).  Frames are cut into chunks of <= max_frames and pipelined
 *      over n_lanes streams so that H2D(i+1), kernels(i) and D2H(i-1) overlap.  Host
 *      buffers that are not pinned are pinned for the duration of the call.
 *      h_hconj / h_hsqrd / h_bits may be NULL.  Synchronous: results are ready on return. */
int lsmrc_demod_frames_host(lsmrc_handle h, const void *h_rx, int n_frames, void *h_hconj,
                            void *h_hsqrd, void *h_combined, void *h_bits);

/* ---- wire-format ingest (SURVEY 8f rank 1, the producer side; not in the reference).  The reference's receive program asks
 *      UHD for cpu format "fc32" over wire format "sc16" (rx_and_corr.cpp:283): the radio's int16 I/Q samples are converted
 *      to complex float ON THE HOST (fc32 = sc16 * scale; UHD's default full scale gives scale = 1/32767) and every sample
 *      then crosses PCIe as 8 bytes.  Host-fed operation is PCIe-bound, so these calls take the wire format itself --
 *      h_rx_iq [F][S][A][N+C][2] int16, 4 bytes per sample -- and convert on the device after the copy: half the bytes on
 *      the link.  int16 -> float is exact and the product rounds once, so the receiver sees bit-for-bit the floats the host
 *      conversion would have produced; everything else is lsmrc_demod_frames_host. */
int lsmrc_demod_frames_host_sc16(lsmrc_handle h, const int16_t *h_rx_iq, int n_frames, float scale, void *h_hconj,
                                 void *h_hsqrd, void *h_combined, void *h_bits);
/* The conversion alone, device to device: out[r][n] = (float)in[r][skip + n] * scale for `rows` rows of row_len_in int16
 * I/Q pairs, keeping row_len_out samples from position `skip` (e.g. skip = C, row_len_out = N drops the cyclic prefix);
 * d_out is complex64 [rows][row_len_out]. */
int lsmrc_sc16_to_fc32_device(lsmrc_handle h, const int16_t *d_iq, long long rows, int row_len_in, int skip, int row_len_out,
                              float scale, void *d_out);

/* ---- per-symbol entry points (replace gpuLS::firstVector gpuLS.cu:351 and
 *      gpuLS::demodOneSymbol :410).  rx_sym is one ring slot [A][N+C]; on_device says
 *      where it lives.  The channel estimate stays inside the handle between calls. ---- */
int lsmrc_first_vector(lsmrc_handle h, const void *rx_sym, int on_device);
int lsmrc_demod_one_symbol(lsmrc_handle h, const void *rx_sym, int on_device,
                           void *h_combined /* K complex64, host */, void *h_bits /* row bytes, host, may be NULL */);
int lsmrc_get_channel(lsmrc_handle h, void *h_hconj /* [A][K] */, void *h_hsqrd /* [K] */);
/* same, into caller-owned DEVICE buffers: the dH / Hsqrd arguments of gpuLS::firstVector
 * (gpuLS.cu:351), which the reference leaves filled for the caller.  Either may be NULL. */
int lsmrc_get_channel_device(lsmrc_handle h, void *d_hconj /* [A][K] */, void *d_hsqrd /* [K] */);

/* ---- streaming ingest from a pinned ring (replaces ShMemSymBuff::readNextSymbolCUDA /
 *      readLastSymbolCUDA, ShMemSymBuff_gpu.hpp:373-445, plus the demod calls that follow
 *      them).  One "lane" = one stream + device staging for one frame + pinned result
 *      buffers.  submit() enqueues H2D of the frame's S slots (slot s at
 *      h_slots + s*slot_stride_bytes), both kernels and the D2H of the results, and
 *      returns at once; wait() blocks until that lane is done and hands back pointers to
 *      the lane's pinned result buffers (valid until the lane is submitted again). ------ */
int lsmrc_ring_submit_frame(lsmrc_handle h, int lane, const void *h_slots, size_t slot_stride_bytes);
/* Allocates the lanes (streams, device staging, pinned result buffers) now instead of inside the first submission --
 * tens of milliseconds of cudaMalloc / cudaMallocHost that a streaming consumer wants behind it before frames arrive. */
int lsmrc_ring_prepare(lsmrc_handle h);
/* one frame that wraps around the end of the ring: n_first slots at h_first, the other S - n_first at h_second */
int lsmrc_ring_submit_split(lsmrc_handle h, int lane, const void *h_first, int n_first,
                            const void *h_second);
/* Several consecutive frames of the ring in one submission (n_frames <= max_frames): n_first slots at h_first, the
 * remaining n_frames*S - n_first at h_second (ring wrap).  Small frames are launch-latency bound; batching the frames
 * that are already waiting in the ring amortises the launch.  lsmrc_ring_wait then returns n_frames results back to
 * back in the lane's buffers. */
int lsmrc_ring_submit_frames(lsmrc_handle h, int lane, const void *h_first, int n_first, const void *h_second, int n_frames);
int lsmrc_ring_wait(lsmrc_handle h, int lane, const void **combined, const void **bits,
                    const void **hconj);
/* blocks until the lane's H2D (or, for frames read in place, the kernel) has finished: its ring slots may be reused */
int lsmrc_ring_copy_done(lsmrc_handle h, int lane);
/* non-blocking form: 1 when the slots of the frame last submitted to `lane` may be reused, 0 when not yet */
int lsmrc_ring_copy_query(lsmrc_handle h, int lane);
/* Timeline of the submission last collected from `lane` (after lsmrc_ring_wait), CUDA-event milliseconds since the
 * handle's first ring submission: ms4[0] submission enqueued (H2D starts when the lane's stream reaches it), [1] H2D
 * finished / slots free, [2] kernels finished, [3] results on the host.  Evidence for the overlap of the three phases
 * across lanes (replaces the clock() timers of ShMemSymBuff_gpu.hpp:373-445). */
int lsmrc_ring_trace(lsmrc_handle h, int lane, float *ms4);

/* ---- stand-alone steps: the individually callable kernel wrappers of gpuLS.cuh:87-99.  The fused
 *      entry points above never go through them; they produce the same intermediate tensors the
 *      reference's wrappers do, for callers that drive the chain step by step.  DEVICE pointers,
 *      enqueued on the compute stream.  A = n_ant, N = fft_size, K = N-1. ------------------------- */
/* DropPrefix (gpuLS.cu:143-156,268-271): out[r][n] = in[r][n + cp], in [rows][N+C] -> out [rows][N] */
int lsmrc_stage_drop_prefix(lsmrc_handle h, void *d_out, const void *d_in, long long rows);
/* batchedFFT (gpuLS.cu:343-349): in-place forward N-point DFT of `rows` rows [rows][N] */
int lsmrc_stage_fft(lsmrc_handle h, void *d_rows, long long rows);
/* FindLeastSquaresGPU / findHs (gpuLS.cu:158-182,273-276): hconj[a][k] = conj(yfft[a][k+1] / X[a][k]);
 * d_x is the reference's replicated pilot [A][K] in bin order, or NULL for the handle's pilot */
int lsmrc_stage_find_hs(lsmrc_handle h, const void *d_yfft, void *d_hconj, const void *d_x);
/* FindHsqrdforMRC / findDistSqrd (gpuLS.cu:185-209,278-282): hsqrd[k] = sum_a |hconj[a][k]|^2 */
int lsmrc_stage_find_hsqrd(lsmrc_handle h, const void *d_hconj, void *d_hsqrd);
/* MultiplyWithChannelConj (gpuLS.cu:212-233,284-287): yf[s][a][k] = yfft[s][a][k+1] * hconj[a][k] */
int lsmrc_stage_mult_conj(lsmrc_handle h, const void *d_yfft, const void *d_hconj, void *d_yf, int n_syms);
/* CombineForMRC (gpuLS.cu:236-259,289-293): out[s][k] = sum_a yf[s][a][k] / hsqrd[k]; out must not
 * alias yf (the reference writes in place and races between blocks) */
int lsmrc_stage_combine(lsmrc_handle h, const void *d_yf, const void *d_hsqrd, void *d_out, int n_syms);
/* ShiftOneRow (gpuLS.cu:109-125,263-266): out[r][i] = in[r][(i + (K-1)/2) mod K], rows of K */
int lsmrc_stage_shift_rows(lsmrc_handle h, const void *d_in, void *d_out, long long rows);
int lsmrc_copy_device(lsmrc_handle h, void *d_dst, const void *d_src, size_t bytes); /* D2D on the compute stream */

/* ---- receive front end before the hot path (SURVEY 8f, rank 1): frame sync and frame stitching of
 *      rx_and_corr.cpp:332-393 + the slot gather of :64-87, on the GPU, so a capture that is already in
 *      device memory never goes back through the CPU correlator and the shm ring. ------------------------ */
/* PN correlator (rx_and_corr.cpp:335-360): metric[ch][i] = |sum_j pn[j]*buf[ch][i+j]| / pn_len over
 * d_buf [n_chan][samps]; *offset = first i (channels scanned in order) with metric >= thres, or -1.
 * d_metric_all (device, [n_chan][samps] float) is optional.  Synchronous. */
int lsmrc_sync_correlate(lsmrc_handle h, const void *d_buf, int n_chan, int samps, const void *d_pn, int pn_len,
                         float thres, int *offset, int *chan, float *metric, void *d_metric_all);
/* Stitch one frame that starts at buf1[ch][offset + pn_len] and wraps into buf2 (rx_and_corr.cpp:372-393)
 * straight into the hot path's input layout [S][A][N+C] (CP left in).  Buffers are [A][samps]. */
int lsmrc_sync_assemble(lsmrc_handle h, const void *d_buf1, const void *d_buf2, int samps, int offset, int pn_len,
                        void *d_rx_frame);

/* ---- multi-user zero forcing (SURVEY 8f rank 4; replaces createZeroForcingMatrix cpuLS.hpp:415-447 with rotCube
 *      :400-413, and multiplyWithChannelInv :449-463 -- defined but never called in the reference; they need
 *      CBLAS/LAPACK there).  Independent of the handle's receiver dimensions; device pointers, complex64.
 *      d_x   [n_users][n_ant][n_sc]  per-user channel, the argument createZeroForcingMatrix takes before rotCube
 *      d_hzf [n_sc][n_users][n_ant]  per subcarrier Hk = Xk^H inv(Xk Xk^H), n_ant x n_users column-major (ld = n_ant)
 *      n_singular (host, may be NULL): subcarriers whose Gram matrix was singular -- a pivot below 1e-6 of its
 *      largest entry -- (their block is zero); passing it makes the call synchronous.  n_users <= 16 and <= n_ant.
 *      lsmrc_zf_apply: d_xd [n_users][n_sc] user symbols -> d_hx [n_ant][n_sc], hx[a][k] = sum_u Hk[a][u] xd[u][k]. */
int lsmrc_zf_create(lsmrc_handle h, const void *d_x, int n_ant, int n_sc, int n_users, void *d_hzf, int *n_singular);
int lsmrc_zf_apply(lsmrc_handle h, const void *d_hzf, const void *d_xd, int n_ant, int n_sc, int n_users, void *d_hx);

/* ---- multi-user uplink: per-user LS channel estimates and linear detection fused with the row FFT (not in the
 *      reference; DESIGN.md 8e, 8h).  Frame format: the usual rx [F][S][A][N+C] (N+C per antenna row, CP first), with
 *      U = n_users and P pilot symbols, in one of two pilot layouts chosen per handle with lsmrc_set_mu_pilots:
 *      LSMRC_MU_PILOTS_TIME (default), P = U:
 *        symbols 0 .. U-1   time-orthogonal pilots: on symbol u user u sends the handle's pilot (lsmrc_set_pilot*),
 *                           the other users are silent;
 *        symbols U .. S-1   data of all U users on the same subcarriers at once.
 *      LSMRC_MU_PILOTS_COMB, P = 1:
 *        symbol 0           comb pilots: user u sends the handle's pilot X[i] on the ascending-frequency indices
 *                           i = u (mod U) (i = 0 .. K-1, the lsmrc_set_pilot order) and nothing on the others;
 *        symbols 1 .. S-1   data of all U users on the same subcarriers at once.
 *      With U = 1 both are the single-user frame.  Per frame f and subcarrier k (FFT-bin order):
 *        H[u][a][k] = Z_u[a][k] / X[k]                       time: LS per user (Z_u: FFT of pilot symbol u)
 *        H[u][a][k] = interpolated LS of symbol 0            comb: LS[a][i] = conj(Z_0[a][i] / X[i]) (conj(H)) is
 *                                                            copied on u's own pilots; between u's nearest pilots
 *                                                            p0 < i < p1 it is LS[p0] + w (LS[p1] - LS[p0]) with
 *                                                            w = (phi(i) - phi(p0)) / (phi(p1) - phi(p0)), fp32;
 *                                                            beyond u's outermost pilot the nearest one is held.
 *                                                            phi(i) = i - N/2 (i < N/2), i - N/2 + 1 (i >= N/2): the
 *                                                            signed frequency, DC skipped.
 *        G_k = H_k^H H_k + lambda I,  W_k = inv(G_k) H_k^H    H_k the A x U matrix; W_k is U x A
 *        xhat[s][u][k] = sum_a W_k[u][a] Z_s[a][k]           every data symbol s
 *      ZF: lambda = 0.  MMSE: lambda = noise_var, the noise variance per antenna and subcarrier after the FFT (same
 *      convention as lsmrc_demod_frames_device_soft).  A subcarrier whose Gram matrix G_k is singular (a pivot below
 *      1e-6 of its largest entry, the rule of lsmrc_zf_create) gets W_k = 0, so its outputs are zero.
 *      With U = 1 and ZF, W = conj(H) / sum_a |H|^2: MRC.
 *      Device pointers, complex64 unless noted; the handle's compute stream, as lsmrc_demod_frames_device:
 *        d_hconj    [F][U][A][K]        conj(H) per user in the reference layout (bin k+1 at index k); may be NULL
 *        d_combined [F][S-P][U][K]      xhat, ascending frequency ([F][S-U][U][K] time, [F][S-1][U][K] comb)
 *        d_bits     [F][S-P][U][row]    hard-demapped xhat, row = lsmrc_bits_row_bytes(N, b); may be NULL
 *        n_singular (host, may be NULL; non-NULL makes the call synchronous): (frame, subcarrier) pairs whose Gram
 *                   matrix was singular.
 *      Any FFT size the handle supports, A <= 256, 1 <= U <= 16, U <= A; time pilots need U < S, comb pilots S >= 2
 *      (U >= S is valid there, e.g. 16 users in 14 symbols).  LSMRC_ERR_INVALID for a bad U or S, an unknown
 *      detector, or MMSE with a noise_var that is not finite and > 0; LSMRC_ERR_NO_PILOT without a pilot.
 *      Nothing is mirrored on the host: with n_singular == NULL the call can be captured into a CUDA graph after one
 *      ordinary call of the same size (which allocates its scratch). */
enum { LSMRC_DETECT_ZF = 0, LSMRC_DETECT_MMSE = 1 };
enum { LSMRC_MU_PILOTS_TIME = 0, LSMRC_MU_PILOTS_COMB = 1 };
/* pilot layout of lsmrc_demod_frames_device_mu and _mu_soft on this handle: LSMRC_MU_PILOTS_TIME (the default) or
 * LSMRC_MU_PILOTS_COMB; any other value is LSMRC_ERR_INVALID.  A call reads it when it is enqueued, so a captured
 * CUDA graph keeps the layout it was captured with. */
int lsmrc_set_mu_pilots(lsmrc_handle h, int layout);
int lsmrc_demod_frames_device_mu(lsmrc_handle h, const void *d_rx, int n_frames, int n_users, int detector,
                                 float noise_var, void *d_hconj, void *d_combined, void *d_bits, int *n_singular);

/* ---- multi-user uplink with soft output: lsmrc_demod_frames_device_mu plus per-user post-detection SINR and max-log
 *      LLRs for a channel decoder (DESIGN.md 8f).  Per frame, subcarrier k and user u, with M_k = inv(G_k) (G_k as
 *      above) and d = [M_k]_uu, sigma2 = noise_var:
 *        ZF:    rho = 1 / (sigma2 d)                      LLRs of xhat
 *        MMSE:  rho = 1 / (lambda d) - 1 (at least 0)     LLRs of xhat / beta, beta = 1 - lambda d = [W_k H_k]_uu
 *                                                         (the MMSE output is biased: xhat = beta x + interference + noise)
 *      rho is the post-detection SINR of user u on subcarrier k; the LLRs are those of lsmrc_demod_frames_device_soft
 *      with sum|H|^2 / noise_var replaced by rho.  A singular subcarrier gets rho = 0 and all-zero LLRs.  With U = 1
 *      both detectors give lsmrc_demod_frames_device_soft's LLRs for the same noise_var.
 *        d_llr      [F][S-P][U][K][b] float, ascending frequency, bit order of the packed bits, LLR > 0 <=> bit 0
 *                   (P pilot symbols: [F][S-U][U][K][b] with time pilots, [F][S-1][U][K][b] with comb pilots)
 *        d_sinr     [F][U][K] float, ascending frequency: rho; may be NULL
 *      Every other argument keeps its meaning and layout from lsmrc_demod_frames_device_mu, and d_combined and d_bits
 *      are byte-identical to what that call writes for the same input.  For MMSE they therefore stay the biased xhat:
 *      only the two sign bits of each symbol are guaranteed to agree with the hard bits, the amplitude bits of the LLRs
 *      come from the unbiased xhat / beta.
 *      noise_var must be finite and > 0 for both detectors (ZF scales its LLRs by it).  LSMRC_ERR_INVALID for a NULL
 *      d_llr or such a noise_var, otherwise the errors of lsmrc_demod_frames_device_mu.  With n_singular == NULL the
 *      call can be captured into a CUDA graph after one ordinary call of the same size. */
int lsmrc_demod_frames_device_mu_soft(lsmrc_handle h, const void *d_rx, int n_frames, int n_users, int detector,
                                      float noise_var, void *d_hconj, void *d_combined, void *d_bits,
                                      void *d_llr, void *d_sinr, int *n_singular);

/* ---- multi-user downlink: zero-forcing precoding from the uplink channel estimates, fused with the inverse row FFT
 *      and cyclic-prefix insertion (DESIGN.md 8g; replaces createZeroForcingMatrix -> multiplyWithChannelInv ->
 *      modOneSymbol -> addPrefix, cpuLS.hpp:391-529, uncalled in the reference).  Channel reciprocity (TDD): the
 *      downlink channel from the antennas to user u is row u of H_k^T, H_k the A x U uplink channel of subcarrier k.
 *      Per frame f and subcarrier k (FFT-bin order):
 *        P_k = conj(H_k) inv(H_k^T conj(H_k) + reg I)        A x U precoder; P_k[a][u] = W_k[u][a], the uplink detector
 *        z[d][a][k] = sum_u P_k[a][u] s[d][u][k]             bin 0 is 0
 *        g_f = sqrt(U K / sum_k |P_k|_F^2)                   one gain per frame: unit-energy symbols give a mean transmit
 *                                                            energy of U per used subcarrier
 *        tx[d][a][C + n] = g_f IDFT(z[d][a])[n]              with the 1/N of numpy.fft.ifft; tx[d][a][0..C) = tx[d][a][N..N+C)
 *      reg = 0 is ZF (H_k^T P_k = I: user u receives g_f s_u), reg > 0 regularised ZF.  A subcarrier whose Gram matrix is
 *      singular (the rule of lsmrc_demod_frames_device_mu) gets P_k = 0 and adds nothing to the power sum; a frame with
 *      no regular subcarrier gets g_f = 0.  The receiver's FFT of a tx row (CP dropped) gives back g_f z.
 *      Device pointers, complex64 unless noted; the handle's compute stream, as lsmrc_demod_frames_device:
 *        d_hconj    [F][U][A][K]          conj(H) per user in the reference layout, as lsmrc_demod_frames_device_mu writes
 *                                         it (the handle keeps no channel state: the caller passes it back)
 *        d_sym      [F][Sd][U][K]         user symbols, ascending frequency (the layout of that call's d_combined)
 *        d_tx       [F][Sd][A][N+C]       time-domain antenna samples, CP first (the receiver's input layout)
 *        d_gain     [F] float             g_f; may be NULL
 *        n_singular (host, may be NULL; non-NULL makes the call synchronous): (frame, subcarrier) pairs whose Gram
 *                   matrix was singular.
 *      A, N and C come from the handle; any FFT size the handle supports, C <= N, A <= 256, 1 <= U <= 16, U <= A,
 *      Sd = n_sym_dl >= 1.  No pilot is needed.  LSMRC_ERR_INVALID for a bad U or Sd, a reg that is not finite and >= 0,
 *      or a NULL d_hconj / d_sym / d_tx; nothing is launched then.  With n_singular == NULL the call can be captured
 *      into a CUDA graph after one ordinary call of the same size (which allocates its scratch). */
int lsmrc_precode_frames_device(lsmrc_handle h, const void *d_hconj, int n_frames, int n_users, float reg,
                                const void *d_sym, int n_sym_dl, void *d_tx, void *d_gain, int *n_singular);

/* ---- memory and stream plumbing, so callers need no CUDA headers (replaces the raw
 *      cudaMalloc/cudaMemcpy/cudaFree calls of gpuLS_main.cu:73-91,135-139) ------------ */
int lsmrc_dev_alloc(lsmrc_handle h, size_t bytes, void **d_ptr);
int lsmrc_dev_free(lsmrc_handle h, void *d_ptr);
int lsmrc_copy_to_device(lsmrc_handle h, void *d_dst, const void *h_src, size_t bytes);
int lsmrc_copy_to_host(lsmrc_handle h, void *h_dst, const void *d_src, size_t bytes);
int lsmrc_host_alloc(lsmrc_handle h, size_t bytes, void **h_ptr); /* pinned */
int lsmrc_host_free(lsmrc_handle h, void *h_ptr);
int lsmrc_host_register(lsmrc_handle h, void *h_ptr, size_t bytes); /* pin an existing mapping (the shm ring) */
int lsmrc_host_unregister(lsmrc_handle h, void *h_ptr);
/* run device-resident calls on a caller stream (NULL = back to the handle's own stream); drains the stream used so
 * far.  A handle is not thread-safe: calls on one handle must come from one thread at a time. */
int lsmrc_set_stream(lsmrc_handle h, void *cuda_stream);
int lsmrc_sync(lsmrc_handle h);
/* Launch policy for whole-frame calls.  A batch small enough to be launch-latency bound (a single small frame,
 * BASELINE config c5) runs as ONE fused kernel -- channel estimate and data symbols together, H kept in shared
 * memory -- instead of the pilot + data pair; lsmrc_demod_frames_host additionally lets that kernel read and write
 * PINNED host buffers in place (no staging copies) when the batch is at most 512 KiB.  enabled: 2 (default) both,
 * 1 fused kernel but staged copies, 0 always the two-kernel path.  Results agree to rounding. */
int lsmrc_set_oneshot(lsmrc_handle h, int enabled);
/* whole-frame calls served by the one-launch kernel so far */
long long lsmrc_oneshot_count(lsmrc_handle h);
/* 2048- and 4096-point receivers, batches of whole frames large enough to fill the GPU: the channel estimate and the data
 * symbols run as ONE persistent launch whose CTAs draw first the pilot work, then the data work from one counter (no drain
 * and ramp between the two phases; data work waits per frame on a device-side ready flag; DESIGN 3.3c).  Results are
 * bit-identical to the kernel pair.  enabled = 0 forces the pair; the count says how many calls took the single launch. */
int lsmrc_set_one_launch_frames(lsmrc_handle h, int enabled);
long long lsmrc_one_launch_frames_count(lsmrc_handle h);

/* ---- instrumentation (replaces the clock() timers of ShMemSymBuff_gpu.hpp:113-257) --- */
/* CUDA-event time of the pilot and data kernels of the most recent lsmrc_demod_frames_device
 * call (waits for them).  Enable with lsmrc_set_timing(h, 1); off by default.  A timed
 * lsmrc_precode_frames_device call reports its two phases in the same places: the precoder build
 * (inverse and gain) as the pilot time, the precode phase (layout pass and precode kernel) as the data time. */
int lsmrc_set_timing(lsmrc_handle h, int enabled);
int lsmrc_last_kernel_ms(lsmrc_handle h, float *pilot_ms, float *data_ms);
/* the same for the most recent min(max_n, 256) timed calls, oldest first; waits for them.  Lets a
 * benchmark read per-kernel durations of a whole timed region without a sync inside it. */
int lsmrc_kernel_ms_history(lsmrc_handle h, int max_n, float *pilot_ms, float *data_ms, int *n_out);
/* number of kernels this library has launched through handle h since creation */
long long lsmrc_launch_count(lsmrc_handle h);
/* plan description, e.g. "N=1024 P=32 R2=32 R3=1 teams=4 threads=128 smem=75512" */
int lsmrc_describe_plan(lsmrc_handle h, char *buf, size_t buf_len);

#ifdef __cplusplus
}
#endif
#endif /* OFDM_LSMRC_H */
