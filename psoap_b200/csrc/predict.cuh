// predict.cuh — the border of the prediction problem (psoap/covariance.py:25-297) and the read-out of its Schur
// complement.  The bordered matrix S = [[K + sigma^2 I, C^T], [C, A]] is built lower triangle only, in the
// factorisation's own layout (column-major, data block front-padded to a tile boundary, border rows after it), the
// leading block is eliminated with the likelihood's kernels, and what is left in the trailing block is
// Sigma = A - C K^-1 C^T while the carried residual holds -C K^-1 (fl - mu).
#pragma once
#include <math_constants.h>

#include "common.cuh"

namespace psoap {

// mode 0: components stacked (predict_f, predict_f_g :81-148, predict_f_g_h :190-251): border index a = c * m + a',
//         A = blockdiag(K_c(predict_c)), C = [K_c(predict_c, data_c)]_c
// mode 1: summed process (predict_f_g_sum :151-187, predict_f_g_h_sum :253-297): A = sum_c K_c(predict_c) + nugget I,
//         C = sum_c K_c(predict_c, data_c)
// mode 2: as 1 with the cross block transposed, C(a, j) = sum_c k_c(data_c[a], predict_c[j]) (the mean of
//         predict_f_g_h_sum multiplies by V12.T, :294; needs m == n)
struct PredictSrc {
    const double* data[3];   // [n] shifted ln-wavelengths of the data, per component
    const double* pred[3];   // [m] prediction grids, per component
    int ncomp, mode;
    int n, m, M;             // M = border size: ncomp * m (mode 0) or m
    int pad, Nn, Nt;         // front padding of the data block, its padded size, total padded size
    double nugget;
    __device__ __forceinline__ double data_z(int c, int j) const { return data[c][j]; }
};

// The chunk farm's source (psoap_farm_predict): the data's ln-wavelengths are the chunk's resident pixels shifted by
// the item's epoch velocities on the fly, z_at(zs, c, j), the very values the data block's fill reads; data[] is unused.
struct PredictFarmSrc : PredictSrc {
    ZSource zs;
    __device__ __forceinline__ double data_z(int c, int j) const { return z_at(zs, c, j); }
};

template <int NCOMP, class Src>
__device__ __forceinline__ double predict_entry(const Src& ps, const double (&amp2)[NCOMP], const double (&p2)[NCOMP],
                                                int a, int c, int ap, int col, const double* __restrict__ etab) {
    // border row a (< M; mode 0: component c, grid point ap) against physical column `col`: a data pixel
    // (pad <= col < Nn) or a border column (col >= Nn)
    if (col < ps.Nn) {
        const int j = col - ps.pad;
        if (j < 0) return 0.0;
        if (ps.mode == 0) return se_term(amp2[c], p2[c], ps.data_z(c, j), ps.pred[c][ap], etab);
        double cov = 0.0;
#pragma unroll
        for (int c = 0; c < NCOMP; ++c) {
            const double t = (ps.mode == 1) ? se_term(amp2[c], p2[c], ps.data_z(c, j), ps.pred[c][a], etab)
                                            : se_term(amp2[c], p2[c], ps.data_z(c, a), ps.pred[c][j], etab);
            cov = (c == 0) ? t : __dadd_rn(cov, t);
        }
        return cov;
    }
    const int b = col - ps.Nn;
    if (b >= ps.M) return 0.0;
    if (ps.mode == 0) {
        const int bp = b - c * ps.m;                      // same component block iff 0 <= bp < m
        if (bp < 0 || bp >= ps.m) return 0.0;
        return se_term(amp2[c], p2[c], ps.pred[c][ap], ps.pred[c][bp], etab);
    }
    double cov = 0.0;
#pragma unroll
    for (int c = 0; c < NCOMP; ++c) {
        const double t = se_term(amp2[c], p2[c], ps.pred[c][a], ps.pred[c][b], etab);
        cov = (c == 0) ? t : __dadd_rn(cov, t);
    }
    return (a == b) ? __dadd_rn(cov, ps.nugget) : cov;
}

// Border rows of S: one CTA per 128 x 128 tile (bi in [Nn/128, Nt/128), bj <= bi), thread = 2 consecutive rows.
// Rows past M (dead padding of the border) get zeros and a unit diagonal; the residual of all border rows is zeroed.
// Src says where the data's ln-wavelengths come from (PredictSrc: per-component arrays; PredictFarmSrc: shifted on the
// fly), as gemm_persistent takes its operand source.
template <int NCOMP, class Src>
__device__ __forceinline__ void predict_border_tile(double* __restrict__ S, int64_t ld, Src ps, GpParams gp,
                                                    double* __restrict__ rvec) {
    __shared__ double etab[64];
    load_exp_table(etab);
    const int Tn = ps.Nn / NB;
    // tile index t -> (bi, bj): rows bi >= Tn, all columns bj <= bi; row bi has bi + 1 tiles
    int t = blockIdx.x, bi = Tn;
    while (t >= bi + 1) { t -= bi + 1; ++bi; }
    const int bj = t;
    double amp2[NCOMP], p2[NCOMP];
#pragma unroll
    for (int c = 0; c < NCOMP; ++c) gp_coeffs(gp, c, amp2[c], p2[c]);
    const int tid = threadIdx.x;
    const int r0 = bi * NB + (tid & 63) * 2;   // physical rows r0, r0 + 1
    const int cg = tid >> 6;
    if (bj == 0 && cg == 0) { rvec[r0] = 0.0; rvec[r0 + 1] = 0.0; }
    int ca[2], apa[2];
#pragma unroll
    for (int e = 0; e < 2; ++e) {
        const int a = r0 + e - ps.Nn;
        ca[e] = (ps.mode == 0 && a < ps.M) ? a / ps.m : 0;
        apa[e] = a - ca[e] * ps.m;
    }
    __syncthreads();
#pragma unroll 2
    for (int cc = 0; cc < 32; ++cc) {
        const int col = bj * NB + cc * 4 + cg;
        double v[2];
#pragma unroll
        for (int e = 0; e < 2; ++e) {
            const int a = r0 + e - ps.Nn;
            if (a >= ps.M) v[e] = (r0 + e == col) ? 1.0 : 0.0;
            else if (col > r0 + e) v[e] = 0.0;               // above the diagonal inside a diagonal tile: never read
            else v[e] = predict_entry<NCOMP>(ps, amp2, p2, a, ca[e], apa[e], col, etab);
        }
        *reinterpret_cast<double2*>(S + r0 + (int64_t)col * ld) = make_double2(v[0], v[1]);
    }
}

template <int NCOMP>
__global__ void __launch_bounds__(256) predict_border_kernel(double* __restrict__ S, int64_t ld, PredictSrc ps, GpParams gp,
                                                             double* __restrict__ rvec) {
    predict_border_tile<NCOMP>(S, ld, ps, gp, rvec);
}

template <int NCOMP>
__global__ void __launch_bounds__(256) predict_border_farm_kernel(double* __restrict__ S, int64_t ld, PredictFarmSrc ps,
                                                                  GpParams gp, double* __restrict__ rvec) {
    predict_border_tile<NCOMP>(S, ld, ps, gp, rvec);
}

// Sigma [M, M] row-major (both triangles) from the lower triangle of the trailing block, delta[a] = -r[Nn + a].
__global__ void predict_readout_kernel(const double* __restrict__ S, int64_t ld, int Nn, int M, const double* __restrict__ rvec,
                                       double* __restrict__ Sigma, double* __restrict__ delta) {
    __shared__ double tile[32][33];
    const int bi = blockIdx.y, bj = blockIdx.x;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;   // 32 x 8
    if (bj > bi) return;
    if (Sigma != nullptr) {
        // read tile (rows 32 bi .., cols 32 bj ..) of the lower triangle, coalesced along rows (column-major)
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int c = bj * 32 + ty + 8 * k, r = bi * 32 + tx;
            tile[ty + 8 * k][tx] = (r < M && c < M && r >= c) ? S[(Nn + r) + (int64_t)(Nn + c) * ld] : 0.0;
        }
        __syncthreads();
        // tile[c][r] = Sigma(r, c) for r >= c.  Write Sigma[r][c] (row-major: coalesced along c) and its mirror.
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int r = bi * 32 + ty + 8 * k, c = bj * 32 + tx;
            if (r < M && c < M && r >= c) Sigma[(int64_t)r * M + c] = tile[tx][ty + 8 * k];
        }
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int c = bj * 32 + ty + 8 * k, r = bi * 32 + tx;   // mirror: Sigma[c][r], coalesced along r
            if (r < M && c < M && r > c) Sigma[(int64_t)c * M + r] = tile[ty + 8 * k][tx];
        }
    }
    if (bj == 0 && delta != nullptr && threadIdx.x < 32) {
        const int a = bi * 32 + threadIdx.x;
        if (a < M) delta[a] = -rvec[Nn + a];
    }
}

// One farm item's outputs from its trailing block: Sigma row-major [M, M] (diag = 0) or its diagonal [M] (diag = 1), and
// delta [M] as predict_readout_kernel writes them.  Every output is NaN when the item's sentinel fired (|v| >= c, a
// negative GP hyper-parameter) or its elimination failed (info != 0): the words grad_flagged reads.  Grid (nb, nb) for
// Sigma, (1, nb) for its diagonal, nb = ceil(M / 32).
__global__ void __launch_bounds__(256) predict_farm_readout_kernel(const double* __restrict__ S, int64_t ld, int Nn, int M,
                                                                   const double* __restrict__ rvec, const int* __restrict__ info,
                                                                   const int* __restrict__ sentinel, int diag,
                                                                   double* __restrict__ Sigma, double* __restrict__ delta) {
    __shared__ double tile[32][33];
    const bool bad = info[0] != 0 || sentinel[0] != 0;
    const int bi = blockIdx.y, bj = blockIdx.x;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;   // 32 x 8
    if (bj > bi) return;
    if (diag) {
        const int a = bi * 32 + threadIdx.x;
        if (threadIdx.x < 32 && a < M) Sigma[a] = bad ? CUDART_NAN : S[(Nn + a) + (int64_t)(Nn + a) * ld];
    } else {
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int c = bj * 32 + ty + 8 * k, r = bi * 32 + tx;
            tile[ty + 8 * k][tx] = (r < M && c < M && r >= c) ? (bad ? CUDART_NAN : S[(Nn + r) + (int64_t)(Nn + c) * ld]) : 0.0;
        }
        __syncthreads();
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int r = bi * 32 + ty + 8 * k, c = bj * 32 + tx;
            if (r < M && c < M && r >= c) Sigma[(int64_t)r * M + c] = tile[tx][ty + 8 * k];
        }
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int c = bj * 32 + ty + 8 * k, r = bi * 32 + tx;
            if (r < M && c < M && r > c) Sigma[(int64_t)c * M + r] = tile[ty + 8 * k][tx];
        }
    }
    if (bj == 0 && threadIdx.x < 32) {
        const int a = bi * 32 + threadIdx.x;
        if (a < M) delta[a] = bad ? CUDART_NAN : -rvec[Nn + a];
    }
}

}  // namespace psoap
