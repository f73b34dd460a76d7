/* layered_oracle.c - sequential C restatement of the layered normalised min-sum decoder (DNALDPC_FLAG_MINSUM |
 * DNALDPC_FLAG_LAYERED, include/dnaldpc.h). Test infrastructure: tests/layered_oracle.py builds and loads it.
 *
 * Written from the contract alone and deliberately unlike the GPU kernels: the layers come from a bitmap first fit,
 * the checks run one after the other (ascending rows inside each layer) and every edge keeps its own c2v message, where
 * the GPU keeps a compressed per-check state (two minima, an index and the signs of v). Build with -ffp-contract=off: every step is one IEEE operation in T. */
#include <math.h>
#include <stdlib.h>
#include <string.h>

/* First fit with one column bitmap per layer. Returns the number of layers. */
int lo_layers(int M, int N, const int *row_ptr, const int *col_idx, int *layer_of_row) {
    unsigned char *used = NULL;
    int L = 0;
    for (int i = 0; i < M; i++) {
        int l = 0;
        for (; l < L; l++) {
            int clash = 0;
            for (int e = row_ptr[i]; e < row_ptr[i + 1] && !clash; e++) clash = used[(size_t)l * N + col_idx[e]];
            if (!clash) break;
        }
        if (l == L) {
            used = (unsigned char *)realloc(used, (size_t)(L + 1) * N);
            memset(used + (size_t)L * N, 0, (size_t)N);
            L++;
        }
        for (int e = row_ptr[i]; e < row_ptr[i + 1]; e++) used[(size_t)l * N + col_idx[e]] = 1;
        layer_of_row[i] = l;
    }
    free(used);
    return M > 0 && L == 0 ? 1 : L;
}

#define LMAX 18446744073709551616.0

#define DEFINE_DECODER(T, NAME)                                                                                          \
    static T clamp_##T(T x) { return x < -(T)LMAX ? -(T)LMAX : (x > (T)LMAX ? (T)LMAX : x); }                           \
    static int syndrome_##T(int M, const int *row_ptr, const int *col_idx, const char *d, char *pchk) {                \
        int c = 0;                                                                                                       \
        for (int i = 0; i < M; i++) {                                                                                    \
            int p = 0;                                                                                                   \
            for (int e = row_ptr[i]; e < row_ptr[i + 1]; e++) p ^= d[col_idx[e]];                                        \
            if (pchk) pchk[i] = (char)p;                                                                                 \
            c += p;                                                                                                      \
        }                                                                                                                \
        return c;                                                                                                        \
    }                                                                                                                    \
    /* One frame. order[M]: rows by ascending layer, ascending row inside a layer. Returns n. */                         \
    static int one_##T(int M, int N, const int *row_ptr, const int *col_idx, const int *order, const double *llr,       \
                       int max_iter, int fixed, T alpha, T *q, T *c2v, T *v, char *d, char *pchk, int *ok, double *post) { \
        for (int j = 0; j < N; j++) {                                                                                    \
            T x = (T)llr[j];                                                                                             \
            if (x != x) x = 0;                                                                                           \
            q[j] = clamp_##T(x);                                                                                         \
            d[j] = !(q[j] > 0);                                                                                          \
        }                                                                                                                \
        for (int e = 0; e < row_ptr[M]; e++) c2v[e] = 0;                                                                 \
        int n = 0;                                                                                                       \
        for (;;) {                                                                                                       \
            const int c = syndrome_##T(M, row_ptr, col_idx, d, NULL);                                                    \
            if (n == max_iter || (c == 0 && !fixed)) break;                                                              \
            for (int r = 0; r < M; r++) {                                                                                \
                const int i = order[r], e0 = row_ptr[i], deg = row_ptr[i + 1] - e0;                                      \
                for (int k = 0; k < deg; k++) v[k] = q[col_idx[e0 + k]] - c2v[e0 + k];                                   \
                /* mu_e = min over the other edges: the second smallest |v| for the (first) smallest one, else the   \
                   smallest; sigma_e = the parity of the other edges' negative v */                                    \
                int first = -1, par = 0;                                                                                 \
                T lo1 = 0, lo2 = 0;                                                                                      \
                for (int m = 0; m < deg; m++) {                                                                          \
                    const T a = fabs(v[m]);                                                                              \
                    par ^= v[m] < 0;                                                                                     \
                    if (first < 0 || a < lo1) { lo2 = lo1; lo1 = a; first = m; }                                         \
                    else if (m == 1 || a < lo2) lo2 = a;                                                                 \
                }                                                                                                        \
                for (int k = 0; k < deg; k++) {                                                                          \
                    const T mu = deg < 2 ? 0 : (k == first ? lo2 : lo1);                                                 \
                    const T mag = alpha * mu;                                                                            \
                    c2v[e0 + k] = (par ^ (v[k] < 0)) ? -mag : mag;                                                       \
                }                                                                                                        \
                for (int k = 0; k < deg; k++) q[col_idx[e0 + k]] = clamp_##T(v[k] + c2v[e0 + k]);                       \
            }                                                                                                            \
            for (int j = 0; j < N; j++) d[j] = !(q[j] > 0);                                                              \
            n++;                                                                                                         \
        }                                                                                                                \
        *ok = syndrome_##T(M, row_ptr, col_idx, d, pchk) == 0;                                                           \
        if (post)                                                                                                        \
            for (int j = 0; j < N; j++) post[j] = (double)q[j];                                                          \
        return n;                                                                                                        \
    }                                                                                                                    \
    /* F frames: llr[F][N] -> iters[F], ok[F], dblk[F][N], pchk[F][M] (may be NULL), post[F][N] (may be NULL). */     \
    void NAME(int M, int N, const int *row_ptr, const int *col_idx, const int *layer_of_row, int n_layers,             \
              const double *llr, int F, int max_iter, int fixed, double alpha, int *iters, char *ok, char *dblk,         \
              char *pchk, double *post) {                                                                                \
        int *order = (int *)malloc(sizeof(int) * (M > 0 ? M : 1));                                                       \
        int r = 0;                                                                                                       \
        for (int l = 0; l < n_layers; l++)                                                                               \
            for (int i = 0; i < M; i++)                                                                                  \
                if (layer_of_row[i] == l) order[r++] = i;                                                                \
        int maxdeg = 1;                                                                                                  \
        for (int i = 0; i < M; i++)                                                                                      \
            if (row_ptr[i + 1] - row_ptr[i] > maxdeg) maxdeg = row_ptr[i + 1] - row_ptr[i];                              \
        T *q = (T *)malloc(sizeof(T) * N), *c2v = (T *)malloc(sizeof(T) * (row_ptr[M] > 0 ? row_ptr[M] : 1));           \
        T *v = (T *)malloc(sizeof(T) * maxdeg);                                                                          \
        for (int f = 0; f < F; f++) {                                                                                    \
            int k = 0;                                                                                                   \
            iters[f] = one_##T(M, N, row_ptr, col_idx, order, llr + (size_t)f * N, max_iter, fixed, (T)alpha, q, c2v,   \
                               v, dblk + (size_t)f * N, pchk ? pchk + (size_t)f * M : NULL, &k,                          \
                               post ? post + (size_t)f * N : NULL);                                                      \
            ok[f] = (char)k;                                                                                             \
        }                                                                                                                \
        free(order); free(q); free(c2v); free(v);                                                                        \
    }

DEFINE_DECODER(double, lo_layered_minsum_decode_f64)
DEFINE_DECODER(float, lo_layered_minsum_decode_f32)
