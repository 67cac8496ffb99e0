/*
 * tests/cpp/mu_soft_oracle.c -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.
 *
 * CPU oracle of the multi-user soft output (lsmrc_demod_frames_device_mu_soft, DESIGN.md 8f), built by
 * tests/test_multi_user_soft.py together with the single-user oracle (oracle/cpuls_oracle.c, oracle/fft_shim.c).
 * It includes the hard multi-user oracle (mu_oracle.c) as its one translation unit, so oracle_demod_frames_mu and the
 * double-precision inverse mz_inv (with the singularity rule of k_zf_create) are the same code in both oracles; build
 * this file instead of mu_oracle.c, not beside it.
 */
#include "mu_oracle.c"

/*
 * Soft output of the multi-user path (lsmrc_demod_frames_device_mu_soft, DESIGN.md 8f), from the hconj [F][U][A][K] and
 * combined [F][S-U][U][K] that oracle_demod_frames_mu wrote.  Per frame and subcarrier M = inv(H^H H + lambda I) again in
 * double (mz_inv, same singularity rule), d = Re M[u][u]:
 *   lambda == 0 (ZF):    rho = 1 / (noise_var d),          scale = 1
 *   lambda > 0  (MMSE):  rho = 1 / (lambda d) - 1 (>= 0),  scale = 1 / (1 - lambda d)
 *   singular, or rho <= 0:  rho = 0, scale = 0
 * sinr [F][U][K] (double, ascending frequency) = rho; llr [F][S-U][U][K][b] = the single-user oracle's fp32 LLR formula
 * (oracle_soft_demap_row) applied to combined * scale with hsqrd := rho (bin order) and noise_var := 1.
 * Returns the number of singular (frame, subcarrier) pairs.
 */
int oracle_mu_soft(const oc_complex *hconj, const oc_complex *combined, int F, int S, int N, int A, int U, int qam_bits, double lambda,
                   double noise_var, double *sinr, float *llr)
{
    const int K = N - 1, D = S - U;
    mz *g = (mz *)malloc(sizeof(mz) * (size_t)U * U);
    mz *aug = (mz *)malloc(sizeof(mz) * (size_t)U * 2 * U);
    double *rho = (double *)malloc(sizeof(double) * (size_t)U * K); /* [U][K] bin order */
    double *scale = (double *)malloc(sizeof(double) * (size_t)U * K);
    float *rho_f = (float *)malloc(sizeof(float) * K);
    oc_complex *row = (oc_complex *)malloc(sizeof(oc_complex) * K);
    int f, u, v, a, k, s, i, bad = 0;
    for (f = 0; f < F; f++) {
        const oc_complex *hc = hconj + (size_t)f * U * A * K;
        for (k = 0; k < K; k++) {
            int ok;
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
            ok = mz_inv(g, U, aug) == 0;
            bad += !ok;
            for (u = 0; u < U; u++) {
                const double d = ok ? g[u * U + u].re : 0.0;
                double r = 0.0, sc = 0.0;
                if (d > 0.0) {
                    if (lambda > 0.0) {
                        r = 1.0 / (lambda * d) - 1.0;
                        if (r > 0.0) sc = 1.0 / (1.0 - lambda * d);
                        else r = 0.0;
                    } else {
                        r = 1.0 / (noise_var * d);
                        sc = 1.0;
                    }
                }
                rho[(size_t)u * K + k] = r;
                scale[(size_t)u * K + k] = sc;
            }
        }
        for (u = 0; u < U; u++) {
            for (k = 0; k < K; k++) {
                const int bin = k + 1, pos = bin < N / 2 ? bin - 1 + N / 2 : bin - N / 2;
                sinr[((size_t)f * U + u) * K + pos] = rho[(size_t)u * K + k];
                rho_f[k] = (float)rho[(size_t)u * K + k];
            }
            for (s = 0; s < D; s++) {
                const size_t orow = ((size_t)f * D + s) * U + u;
                const oc_complex *c = combined + orow * K;
                for (i = 0; i < K; i++) {
                    const double sc = scale[(size_t)u * K + (i + (K - 1) / 2) % K]; /* ascending i -> bin order */
                    row[i].real = (float)(c[i].real * sc);
                    row[i].imag = (float)(c[i].imag * sc);
                }
                oracle_soft_demap_row(row, rho_f, K, qam_bits, 1.0f, llr + orow * K * qam_bits);
            }
        }
    }
    free(g);
    free(aug);
    free(rho);
    free(scale);
    free(rho_f);
    free(row);
    return bad;
}
