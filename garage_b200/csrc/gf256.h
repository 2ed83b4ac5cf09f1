// gf256.h -- GF(2^8)/0x11D arithmetic shared by host (matrix construction) and device
// (table build, decode planning).  Product code: does NOT use anything under oracle/.
//
// Field definition: SURVEY.md section 8(c) / DESIGN.md "Field".  The reference has no
// counterpart (no RS code in deuxfleurs-org/garage); the framing it imposes is cited where
// it matters (rs_kernels.cuh, garage_ec.cu).
#pragma once
#include <stdint.h>

#include "gf256_tables.inc"

#define GARAGE_EC_MAX_K_HOST 32
#define GARAGE_EC_MAX_M_HOST 8

namespace garage_ec {

// host copies
static const uint8_t h_gf_exp[512] = GARAGE_EC_GF_EXP_INIT;
static const uint8_t h_gf_log[256] = GARAGE_EC_GF_LOG_INIT;

inline uint8_t h_mul(uint8_t a, uint8_t b)
{
    return (a && b) ? h_gf_exp[h_gf_log[a] + h_gf_log[b]] : 0;
}
inline uint8_t h_inv(uint8_t a) { return h_gf_exp[255 - h_gf_log[a]]; }

// In-place Gauss-Jordan inversion of an n x n matrix; false if singular.
inline bool h_invert(uint8_t *M, int n)
{
    uint8_t w[GARAGE_EC_MAX_K_HOST * 2 * GARAGE_EC_MAX_K_HOST];
    const int W = 2 * n;
    for (int r = 0; r < n; r++)
        for (int c = 0; c < W; c++) w[r * W + c] = c < n ? M[r * n + c] : (uint8_t)(c - n == r);
    for (int c = 0; c < n; c++) {
        int piv = -1;
        for (int r = c; r < n; r++)
            if (w[r * W + c]) { piv = r; break; }
        if (piv < 0) return false;
        if (piv != c)
            for (int x = 0; x < W; x++) {
                uint8_t t = w[c * W + x];
                w[c * W + x] = w[piv * W + x];
                w[piv * W + x] = t;
            }
        const uint8_t iv = h_inv(w[c * W + c]);
        for (int x = 0; x < W; x++) w[c * W + x] = h_mul(w[c * W + x], iv);
        for (int r = 0; r < n; r++) {
            const uint8_t f = w[r * W + c];
            if (r == c || !f) continue;
            for (int x = 0; x < W; x++) w[r * W + x] ^= h_mul(f, w[c * W + x]);
        }
    }
    for (int r = 0; r < n; r++)
        for (int c = 0; c < n; c++) M[r * n + c] = w[r * W + n + c];
    return true;
}

// Parity rows P (m x k).  kind 0: systematic Vandermonde, V[r][c] = r^c (0^0 = 1),
// P = V[k..k+m) * inv(V[0..k)).  kind 1: Cauchy, P[i][j] = 1/((k+i)^j).
inline bool h_build_matrix(int k, int m, int kind, uint8_t *P)
{
    if (kind == 1) {
        for (int i = 0; i < m; i++)
            for (int j = 0; j < k; j++) P[i * k + j] = h_inv((uint8_t)((k + i) ^ j));
        return true;
    }
    if (kind != 0) return false;
    uint8_t V[(GARAGE_EC_MAX_K_HOST + GARAGE_EC_MAX_M_HOST) * GARAGE_EC_MAX_K_HOST];
    uint8_t T[GARAGE_EC_MAX_K_HOST * GARAGE_EC_MAX_K_HOST];
    for (int r = 0; r < k + m; r++) {
        uint8_t p = 1;
        for (int c = 0; c < k; c++) {
            V[r * k + c] = p;
            p = h_mul(p, (uint8_t)r);
        }
    }
    for (int i = 0; i < k * k; i++) T[i] = V[i];
    if (!h_invert(T, k)) return false;
    for (int i = 0; i < m; i++)
        for (int j = 0; j < k; j++) {
            uint8_t acc = 0;
            for (int x = 0; x < k; x++) acc ^= h_mul(V[(k + i) * k + x], T[x * k + j]);
            P[i * k + j] = acc;
        }
    return true;
}

// Column multipliers of the generalized Reed-Solomon structure of the code [I; P] with evaluation
// points r = 0..k+m-1: v with  sum_r v_r r^l c_r = 0  for every codeword c and l < m.  Written per
// data column j (the codeword e_j + P[:, j]):  v_j j^l + sum_i v_{k+i} (k+i)^l P[i][j] = 0.  The
// k*m x (k+m) system must have a one-dimensional null space with no zero entry; false otherwise
// (a matrix that is not GRS with these points: errors cannot be located with syndromes).
inline bool h_grs_multipliers(int k, int m, const uint8_t *P, uint8_t *v)
{
    const int n = k + m;
    uint8_t A[GARAGE_EC_MAX_K_HOST * GARAGE_EC_MAX_M_HOST][GARAGE_EC_MAX_K_HOST + GARAGE_EC_MAX_M_HOST];
    auto pw = [](uint8_t a, int e) {
        uint8_t r = 1;
        for (int i = 0; i < e; i++) r = h_mul(r, a);
        return r;
    };
    int rows = 0;
    for (int j = 0; j < k; j++)
        for (int l = 0; l < m; l++, rows++) {
            for (int c = 0; c < n; c++) A[rows][c] = 0;
            A[rows][j] = pw((uint8_t)j, l);
            for (int i = 0; i < m; i++) A[rows][k + i] = h_mul(pw((uint8_t)(k + i), l), P[i * k + j]);
        }
    // row echelon form; the null space is one-dimensional iff exactly one column has no pivot
    int piv_of_col[GARAGE_EC_MAX_K_HOST + GARAGE_EC_MAX_M_HOST];
    int r0 = 0, free_col = -1;
    for (int c = 0; c < n; c++) {
        piv_of_col[c] = -1;
        int pr = -1;
        for (int r = r0; r < rows; r++)
            if (A[r][c]) { pr = r; break; }
        if (pr < 0) {
            if (free_col >= 0) return false;  // null space of dimension >= 2
            free_col = c;
            continue;
        }
        for (int x = 0; x < n; x++) {
            const uint8_t t = A[r0][x];
            A[r0][x] = A[pr][x];
            A[pr][x] = t;
        }
        const uint8_t iv = h_inv(A[r0][c]);
        for (int x = 0; x < n; x++) A[r0][x] = h_mul(A[r0][x], iv);
        for (int r = 0; r < rows; r++) {
            const uint8_t f = A[r][c];
            if (r == r0 || !f) continue;
            for (int x = 0; x < n; x++) A[r][x] ^= h_mul(f, A[r0][x]);
        }
        piv_of_col[c] = r0++;
    }
    if (free_col < 0) return false;  // only the zero vector: not a GRS code with these points
    // reduced form: v_c = A[piv][free] * v_free for pivot columns (characteristic 2), v_free = 1
    for (int c = 0; c < n; c++) {
        v[c] = c == free_col ? 1 : A[piv_of_col[c]][free_col];
        if (!v[c]) return false;
    }
    return true;
}

}  // namespace garage_ec
