// grad.cuh — gradient of the log-likelihood with respect to the GP hyper-parameters, the mean and the shifted
// ln-wavelengths (and, through the per-epoch sum and the orbit Jacobian, the orbital parameters).
//
//   dlnlike/dtheta = 1/2 sum_ij W_ij dK_ij/dtheta,   W = alpha alpha^T - K^-1,   alpha = K^-1 (fl - mu)
//
// K^-1 and alpha come from the factorisation itself: the data block of the bordered matrix [[K, I], [I, 0]] (border
// = the identity in data order) is eliminated with the likelihood's kernels (api.cu launch_factor, restricted to the
// rows the identity border can reach), which leaves -K^-1 in the trailing block and -alpha in the carried residual.
// The contraction then recomputes the covariance terms with the fill's own arithmetic (z_at, gp_coeffs, exp_neg).
// Every sum runs in a fixed order (per-tile partials, then fixed-order reductions): the gradient is bit-identical from
// run to run, like the likelihood.  No floating-point atomics.
#pragma once
#include <math_constants.h>

#include "common.cuh"
#include "orbit.cuh"

namespace psoap {

// Border rows [Nn, Nt) of the identity-bordered matrix S (column-major, leading dimension ld): lower triangle of
// row Nn + a is 1 at column pad + a (data index a) for a < N, and the unit diagonal on the dead rows a >= N; the
// carried residual of the border rows starts at zero.  One CTA per 128 x 128 border tile (bi >= Tn, bj <= bi),
// thread = 2 consecutive rows, as predict_border_kernel.
__global__ void __launch_bounds__(256) grad_border_kernel(double* __restrict__ S, int64_t ld, int Nn, int N, int pad,
                                                          double* __restrict__ rvec) {
    const int Tn = Nn / NB;
    int t = blockIdx.x, bi = Tn;
    while (t >= bi + 1) { t -= bi + 1; ++bi; }
    const int bj = t;
    const int tid = threadIdx.x;
    const int r0 = bi * NB + (tid & 63) * 2;
    const int cg = tid >> 6;
    if (bj == 0 && cg == 0) { rvec[r0] = 0.0; rvec[r0 + 1] = 0.0; }
#pragma unroll 4
    for (int cc = 0; cc < 32; ++cc) {
        const int col = bj * NB + cc * 4 + cg;
        double v[2];
#pragma unroll
        for (int e = 0; e < 2; ++e) {
            const int a = r0 + e - Nn;
            const int one = (a < N) ? pad + a : r0 + e;
            v[e] = (col == one) ? 1.0 : 0.0;
        }
        *reinterpret_cast<double2*>(S + r0 + (int64_t)col * ld) = make_double2(v[0], v[1]);
    }
}

// Where the contraction writes: per lower tile t of the trailing block, 2 NCOMP scalars
//   tile[t][2c]     = sum_{a>b in tile} W_ab e_c,ab + 1/2 sum_{a in diagonal tile} W_aa       (e = exp(p2 Delta^2))
//   tile[t][2c + 1] = sum_{a>b in tile} W_ab k_c,ab (p2 Delta^2)
// and per pair of 128-blocks (I, J) the partial pixel sums slot[(I * Tb + J) * NCOMP + c][128] of
//   g_c,a = sum_b W_ab k_c,ab (zeta_a - zeta_b)   (dlnlike/dzeta_c,a = 2 p2_c g_c,a)
// from tile (I, J) (rows, J <= I) or tile (J, I) (columns, J > I); the diagonal tile sums both.
struct GradOut {
    double* tile;
    double* slot;
    int Tb;
};

template <int NCOMP>
__global__ void __launch_bounds__(256) lnlike_grad_kernel(const double* __restrict__ S, int64_t ld, int Nn, int N,
                                                          const double* __restrict__ rvec, ZSource zs, GpParams gp,
                                                          GradOut out) {
    const int t = blockIdx.x;
    int bi = (int)((sqrtf(8.0f * (float)t + 1.0f) - 1.0f) * 0.5f);
    while ((bi + 1) * (bi + 2) / 2 <= t) ++bi;
    while (bi * (bi + 1) / 2 > t) --bi;
    const int bj = t - bi * (bi + 1) / 2;
    __shared__ double zj[NCOMP][NB];
    __shared__ double alj[NB];
    __shared__ double etab[64];
    __shared__ double colp[NCOMP][2][4][32];   // [c][warp of the column group][column group][column]
    __shared__ double rowp[NCOMP][4][NB];      // [c][column group][row]
    __shared__ double red[2 * NCOMP][8];
    load_exp_table(etab);
    const int tid = threadIdx.x;
    if (tid < NB) {
        const int b = bj * NB + tid;
#pragma unroll
        for (int c = 0; c < NCOMP; ++c) zj[c][tid] = (b < N) ? z_at(zs, c, b) : 0.0;
        alj[tid] = (b < N) ? -rvec[Nn + b] : 0.0;
    }
    double amp2[NCOMP], p2[NCOMP];
#pragma unroll
    for (int c = 0; c < NCOMP; ++c) gp_coeffs(gp, c, amp2[c], p2[c]);
    const int a0 = bi * NB + (tid & 63) * 2;
    double zi[NCOMP][2], ali[2];
#pragma unroll
    for (int e = 0; e < 2; ++e) {
#pragma unroll
        for (int c = 0; c < NCOMP; ++c) zi[c][e] = (a0 + e < N) ? z_at(zs, c, a0 + e) : 0.0;
        ali[e] = (a0 + e < N) ? -rvec[Nn + a0 + e] : 0.0;
    }
    __syncthreads();
    const int cg = tid >> 6, lane = tid & 31, wg = (tid >> 5) & 1;
    const double* base = S + Nn + (int64_t)Nn * ld;
    double sA[NCOMP], sB[NCOMP], rg[NCOMP][2];
#pragma unroll
    for (int c = 0; c < NCOMP; ++c) { sA[c] = 0.0; sB[c] = 0.0; rg[c][0] = 0.0; rg[c][1] = 0.0; }
    const bool diag = (bi == bj);
#pragma unroll 2
    for (int cc = 0; cc < 32; ++cc) {
        const int jl = cc * 4 + cg;
        const int b = bj * NB + jl;
        const double2 m = *reinterpret_cast<const double2*>(base + a0 + (int64_t)b * ld);
        const double mk[2] = {m.x, m.y};
        double cgsum[NCOMP];
#pragma unroll
        for (int c = 0; c < NCOMP; ++c) cgsum[c] = 0.0;
#pragma unroll
        for (int e = 0; e < 2; ++e) {
            const int a = a0 + e;
            // W_ab = alpha_a alpha_b - K^-1_ab below the diagonal; on it 1/2 W_aa, whose covariance term has
            // Delta = 0: exp_neg(0) = 1 enters the amp sums and nothing else (x = 0, r = 0)
            const bool live = (a < N) && (b < N) && (!diag || a >= b);
            const double wab = fma(ali[e], alj[jl], mk[e]);
            const double w = live ? ((diag && a == b) ? 0.5 * wab : wab) : 0.0;
#pragma unroll
            for (int c = 0; c < NCOMP; ++c) {
                const double r = __dsub_rn(zj[c][jl], zi[c][e]);
                const double x = __dmul_rn(__dmul_rn(p2[c], r), r);
                const double ex = exp_neg(x, etab);
                const double wk = w * __dmul_rn(amp2[c], ex);
                sA[c] = fma(w, ex, sA[c]);
                sB[c] = fma(wk, x, sB[c]);
                const double g = wk * r;                                  // W k (zeta_b - zeta_a)
                rg[c][e] -= g;
                cgsum[c] += g;
            }
        }
        // column partial of b: 64 threads (2 warps) hold its 128 rows
#pragma unroll
        for (int c = 0; c < NCOMP; ++c) {
            double v = cgsum[c];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
            if (lane == 0) colp[c][wg][cg][cc] = v;
        }
    }
#pragma unroll
    for (int c = 0; c < NCOMP; ++c) {
        rowp[c][cg][a0 - bi * NB] = rg[c][0];
        rowp[c][cg][a0 - bi * NB + 1] = rg[c][1];
    }
    // tile scalars: warp butterfly, then the 8 warps in order
#pragma unroll
    for (int c = 0; c < NCOMP; ++c) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            sA[c] += __shfl_xor_sync(0xffffffffu, sA[c], o);
            sB[c] += __shfl_xor_sync(0xffffffffu, sB[c], o);
        }
        if (lane == 0) { red[2 * c][tid >> 5] = sA[c]; red[2 * c + 1][tid >> 5] = sB[c]; }
    }
    __syncthreads();
    if (tid < 2 * NCOMP) {
        double s = 0.0;
#pragma unroll
        for (int w = 0; w < 8; ++w) s += red[tid][w];
        out.tile[(int64_t)t * 2 * NCOMP + tid] = s;
    }
    if (tid < NB) {
        const int r = tid;
#pragma unroll
        for (int c = 0; c < NCOMP; ++c) {
            const double rowsum = ((rowp[c][0][r] + rowp[c][1][r]) + rowp[c][2][r]) + rowp[c][3][r];
            // column r of the tile: group r % 4, entry r / 4, two warps
            const double colsum = colp[c][0][r & 3][r >> 2] + colp[c][1][r & 3][r >> 2];
            if (diag) {
                out.slot[((int64_t)(bi * out.Tb + bi) * NCOMP + c) * NB + r] = rowsum + colsum;
            } else {
                out.slot[((int64_t)(bi * out.Tb + bj) * NCOMP + c) * NB + r] = rowsum;
                out.slot[((int64_t)(bj * out.Tb + bi) * NCOMP + c) * NB + r] = colsum;
            }
        }
    }
}

// amp_c, l_c for a component index known only at run time (selects, not a dynamically indexed parameter array: no
// stack frame); p2 as gp_coeffs computes it
__device__ __forceinline__ void gp_pick(const GpParams& gp, int c, double& a, double& l) {
    if (gp.dev) { a = gp.dev[2 * c]; l = gp.dev[2 * c + 1]; return; }
    a = (c == 0) ? gp.amp[0] : (c == 1) ? gp.amp[1] : gp.amp[2];
    l = (c == 0) ? gp.l[0] : (c == 1) ? gp.l[1] : gp.l[2];
}

__device__ __forceinline__ bool grad_flagged(const int* __restrict__ info, const int* __restrict__ sentinel) {
    return info[0] != 0 || (sentinel != nullptr && sentinel[0] != 0);
}

// Hyper-parameter gradient [amp_0, l_0, amp_1, l_1, ..., mu] from the tile partials, in tile order; NaN everywhere
// when the likelihood is -inf (info != 0, or the sentinel of the orbit / hyper-parameter check fired).
__global__ void __launch_bounds__(256) grad_hyp_kernel(const double* __restrict__ tile, int ntiles, int ncomp,
                                                       const double* __restrict__ rvec, int Nn, int N, GpParams gp,
                                                       const int* __restrict__ info, const int* __restrict__ sentinel,
                                                       double* __restrict__ grad_hyp) {
    __shared__ double red[256];
    const int tid = threadIdx.x;
    const bool bad = grad_flagged(info, sentinel);
    for (int q = 0; q <= 2 * ncomp; ++q) {
        double s = 0.0;
        if (q < 2 * ncomp)
            for (int t = tid; t < ntiles; t += 256) s += tile[(int64_t)t * 2 * ncomp + q];
        else
            for (int a = tid; a < N; a += 256) s -= rvec[Nn + a];   // sum alpha
        red[tid] = s;
        __syncthreads();
        for (int h = 128; h > 0; h >>= 1) {
            if (tid < h) red[tid] += red[tid + h];
            __syncthreads();
        }
        if (tid == 0) {
            double g = red[0];
            if (q < 2 * ncomp) {
                double a, l;
                gp_pick(gp, q >> 1, a, l);
                g = (q & 1) ? -2.0 * g / l : 2.0 * a * g;
            }
            grad_hyp[q] = bad ? CUDART_NAN : g;
        }
        __syncthreads();
    }
}

// dlnlike/dzeta_c,a = 2 p2_c sum_J slot[I][J][c][a % 128] (J in order); block (c, I), 128 threads.
__global__ void __launch_bounds__(128) grad_pixel_kernel(const double* __restrict__ slot, int Tb, int ncomp, int N,
                                                         GpParams gp, const int* __restrict__ info,
                                                         const int* __restrict__ sentinel, double* __restrict__ grad_z) {
    const int c = blockIdx.x % ncomp, I = blockIdx.x / ncomp;
    const int a = I * NB + threadIdx.x;
    if (a >= N) return;
    double s = 0.0;
    for (int J = 0; J < Tb; ++J) s += slot[((int64_t)(I * Tb + J) * ncomp + c) * NB + threadIdx.x];
    double amp, l;
    gp_pick(gp, c, amp, l);
    const double p2 = __ddiv_rn(-0.5 * C_KMS2, __dmul_rn(l, l));
    grad_z[(int64_t)c * N + a] = grad_flagged(info, sentinel) ? CUDART_NAN : 2.0 * p2 * s;
}

// dlnlike/dv_c[e] = -(1/c_kms) sum_{i : epoch(i) = e} dlnlike/dzeta_c,i; block (c, e), no assumption that an epoch's
// pixels are contiguous.
__global__ void __launch_bounds__(256) grad_epoch_kernel(const double* __restrict__ grad_z, const int32_t* __restrict__ epoch,
                                                         int64_t N, int n_epochs, double* __restrict__ grad_v) {
    __shared__ double red[256];
    const int c = blockIdx.x / n_epochs, e = blockIdx.x % n_epochs;
    const int tid = threadIdx.x;
    double s = 0.0;
    for (int64_t i = tid; i < N; i += 256)
        if (epoch[i] == e) s += grad_z[(int64_t)c * N + i];
    red[tid] = s;
    __syncthreads();
    for (int h = 128; h > 0; h >>= 1) {
        if (tid < h) red[tid] += red[tid + h];
        __syncthreads();
    }
    if (tid == 0) grad_v[blockIdx.x] = -red[0] / C_KMS;
}

// Full registered gradient of one chunk (orbital then GP, utils.registered_params order):
//   grad_p[k < norb] = sum_c sum_e dlnlike/dv_c[e] dv_c[e]/dp_k,  grad_p[norb + j] = grad_hyp[j]  (j < 2 ncomp)
__global__ void grad_chain_kernel(const double* __restrict__ grad_v, const double* __restrict__ jac,
                                  const double* __restrict__ grad_hyp, int ncomp, int n_epochs, int norb,
                                  const int* __restrict__ info, const int* __restrict__ sentinel,
                                  double* __restrict__ grad_p) {
    const int k = threadIdx.x;
    if (k >= norb + 2 * ncomp) return;
    double g;
    if (k < norb) {
        g = 0.0;
        for (int c = 0; c < ncomp; ++c)
            for (int e = 0; e < n_epochs; ++e)
                g = fma(grad_v[c * n_epochs + e], jac[((int64_t)c * n_epochs + e) * norb + k], g);
    } else {
        g = grad_hyp[k - norb];
    }
    grad_p[k] = grad_flagged(info, sentinel) ? CUDART_NAN : g;
}

// -inf likelihood found on the host (negative hyper-parameters): NaN in every gradient entry.
__global__ void grad_fill_kernel(double* __restrict__ out, int64_t n, double v) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) out[i] = v;
}

__global__ void orbit_jacobian_kernel(int model, const double* __restrict__ p, const double* __restrict__ dates,
                                      int n_epochs, double* __restrict__ jac) {
    orbit_jacobian_block(model, p, dates, n_epochs, jac);
}

}  // namespace psoap
