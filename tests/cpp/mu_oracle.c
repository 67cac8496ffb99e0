/*
 * tests/cpp/mu_oracle.c -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.
 *
 * CPU oracle of the multi-user receive path (lsmrc_demod_frames_device_mu, DESIGN.md 8e), linked with the
 * single-user oracle (oracle/cpuls_oracle.c, oracle/fft_shim.c) and built by tests/test_multi_user.py.
 *   per user u:        LS estimate from pilot symbol u        oracle_first_vector (the single-user pilot path)
 *   per subcarrier k:  G = H^H H + lambda I, inverse           double precision, Gauss-Jordan with partial pivoting and
 *                                                              the singularity rule of oracle/zf_oracle.c / k_zf_create
 *                      W = inv(G) H^H  (U x A)                 double
 *   per data symbol:   xhat[u][k] = sum_a W[u][a] Z[a][k]      double, Z = fp32 FFT of the data symbol (fft_shim)
 *                      ascending-frequency order, hard demap   oracle_shift_one_row, oracle_demap_row
 * Layouts as the C ABI: rx [F][S][A][N+C]; hconj [F][U][A][K]; combined [F][S-U][U][K]; bits [F][S-U][U][row].
 */
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include "../../oracle/cpuls_oracle.h"
#include "../../oracle/fft_shim.h"

typedef struct {
    double re, im;
} mz;
static mz mz_mul(mz a, mz b) { mz r = {a.re * b.re - a.im * b.im, a.re * b.im + a.im * b.re}; return r; }
static mz mz_div(mz a, mz b)
{
    const double d = b.re * b.re + b.im * b.im;
    mz r = {(a.re * b.re + a.im * b.im) / d, (a.im * b.re - a.re * b.im) / d};
    return r;
}

/* inverse of the U x U row-major matrix g in place (Gauss-Jordan, partial pivoting on |re|+|im|); -1 if a pivot is below
 * 1e-6 of the largest entry (the rule of k_zf_create) */
static int mz_inv(mz *g, int U, mz *w)
{
    int i, j, c;
    double gmax = 0.0;
    memset(w, 0, sizeof(mz) * (size_t)U * 2 * U);
    for (i = 0; i < U; i++) {
        for (j = 0; j < U; j++) {
            const double m = fabs(g[i * U + j].re) + fabs(g[i * U + j].im);
            w[i * 2 * U + j] = g[i * U + j];
            if (m > gmax) gmax = m;
        }
        w[i * 2 * U + U + i].re = 1.0;
    }
    for (c = 0; c < U; c++) {
        int p = c;
        double best = -1.0;
        for (i = c; i < U; i++) {
            const double m = fabs(w[i * 2 * U + c].re) + fabs(w[i * 2 * U + c].im);
            if (m > best) {
                best = m;
                p = i;
            }
        }
        if (!(best > 1e-6 * gmax)) return -1;
        if (p != c)
            for (j = 0; j < 2 * U; j++) {
                const mz t = w[c * 2 * U + j];
                w[c * 2 * U + j] = w[p * 2 * U + j];
                w[p * 2 * U + j] = t;
            }
        {
            const mz piv = w[c * 2 * U + c];
            for (j = 0; j < 2 * U; j++) w[c * 2 * U + j] = mz_div(w[c * 2 * U + j], piv);
        }
        for (i = 0; i < U; i++) {
            mz f;
            if (i == c) continue;
            f = w[i * 2 * U + c];
            for (j = 0; j < 2 * U; j++) {
                const mz t = mz_mul(f, w[c * 2 * U + j]);
                w[i * 2 * U + j].re -= t.re;
                w[i * 2 * U + j].im -= t.im;
            }
        }
    }
    for (i = 0; i < U; i++)
        for (j = 0; j < U; j++) g[i * U + j] = w[i * 2 * U + U + j];
    return 0;
}

/* returns the number of singular (frame, subcarrier) pairs; bits may be NULL */
int oracle_demod_frames_mu(const oc_complex *rx, const oc_complex *pilot_asc, int F, int S, int A, int N, int C, int U,
                           int qam_bits, double lambda, oc_complex *hconj, oc_complex *combined, uint8_t *bits)
{
    const int K = N - 1, D = S - U;
    const size_t slot = (size_t)A * (N + C), row_bytes = oracle_bits_row_bytes(K, qam_bits);
    oc_complex *x_bin = (oc_complex *)malloc(sizeof(oc_complex) * K);
    float *hsqrd = (float *)malloc(sizeof(float) * K);
    oc_complex *z = (oc_complex *)malloc(sizeof(oc_complex) * (size_t)A * N);
    mz *w = (mz *)malloc(sizeof(mz) * (size_t)K * U * A); /* [k][u][a] */
    mz *g = (mz *)malloc(sizeof(mz) * (size_t)U * U);
    mz *aug = (mz *)malloc(sizeof(mz) * (size_t)U * 2 * U);
    oc_complex *out = (oc_complex *)malloc(sizeof(oc_complex) * K);
    int f, u, v, a, k, s, bad = 0;
    oracle_pilot_to_bin_order(pilot_asc, x_bin, K);
    for (f = 0; f < F; f++) {
        const oc_complex *fr = rx + (size_t)f * S * slot;
        oc_complex *hc = hconj + (size_t)f * U * A * K; /* [U][A][K] */
        for (u = 0; u < U; u++) oracle_first_vector(fr + (size_t)u * slot, x_bin, hc + (size_t)u * A * K, hsqrd, A, N, C);
        for (k = 0; k < K; k++) {
            mz *wk = w + (size_t)k * U * A;
            /* H[a][u] = conj(hconj[u][a][k]);  G[u][v] = sum_a conj(H[a][u]) H[a][v] = sum_a hconj_u * conj(hconj_v) */
            for (u = 0; u < U; u++)
                for (v = 0; v < U; v++) {
                    mz acc = {u == v ? lambda : 0.0, 0.0};
                    for (a = 0; a < A; a++) {
                        const oc_complex p = hc[((size_t)u * A + a) * K + k], q = hc[((size_t)v * A + a) * K + k];
                        const mz pp = {p.real, p.imag}, qq = {q.real, -q.imag};
                        const mz t = mz_mul(pp, qq);
                        acc.re += t.re;
                        acc.im += t.im;
                    }
                    g[u * U + v] = acc;
                }
            if (mz_inv(g, U, aug) != 0) {
                memset(wk, 0, sizeof(mz) * (size_t)U * A);
                bad++;
                continue;
            }
            /* W[u][a] = sum_v Gi[u][v] conj(H[a][v]) = sum_v Gi[u][v] hconj[v][a][k] */
            for (u = 0; u < U; u++)
                for (a = 0; a < A; a++) {
                    mz acc = {0.0, 0.0};
                    for (v = 0; v < U; v++) {
                        const oc_complex q = hc[((size_t)v * A + a) * K + k];
                        const mz qq = {q.real, q.imag};
                        const mz t = mz_mul(g[u * U + v], qq);
                        acc.re += t.re;
                        acc.im += t.im;
                    }
                    wk[u * A + a] = acc;
                }
        }
        for (s = 0; s < D; s++) {
            const oc_complex *sym = fr + (size_t)(U + s) * slot;
            for (a = 0; a < A; a++)
                oracle_fft_f32(N, (const float *)(sym + (size_t)a * (N + C) + C), (float *)(z + (size_t)a * N), FFTW_FORWARD);
            for (u = 0; u < U; u++) {
                const size_t orow = ((size_t)f * D + s) * U + u;
                for (k = 0; k < K; k++) {
                    const mz *wk = w + (size_t)k * U * A + (size_t)u * A;
                    double re = 0.0, im = 0.0;
                    for (a = 0; a < A; a++) {
                        const oc_complex y = z[(size_t)a * N + k + 1];
                        re += wk[a].re * y.real - wk[a].im * y.imag;
                        im += wk[a].re * y.imag + wk[a].im * y.real;
                    }
                    out[k].real = (float)re;
                    out[k].imag = (float)im;
                }
                oracle_shift_one_row(out, K);
                memcpy(combined + orow * K, out, sizeof(oc_complex) * K);
                if (bits) oracle_demap_row(out, K, qam_bits, bits + orow * row_bytes, NULL);
            }
        }
    }
    free(x_bin);
    free(hsqrd);
    free(z);
    free(w);
    free(g);
    free(aug);
    free(out);
    return bad;
}
