// fill.cuh — squared-exponential covariance fills (replaces psoap/matrix_functions.pyx).
#pragma once
#include "common.cuh"

namespace psoap {

// ------------------------------------------------------------------------------------------------------
// Internal fill: lower triangle of K + sigma^2 I into the factorisation workspace.
//   W: column-major [Np, ld], Np = T*128; data index i lives at physical index i + pad (pad = Np - N,
//   FRONT padding: the first `pad` rows/columns are the identity, so every panel after the first is full).
//   One CTA per 128x128 tile with bi >= bj (1-D grid over the T (T+1) / 2 lower tiles); thread = 2 consecutive rows
//   (double2 stores, 512 B per warp).  Diagonal tiles also initialise the residual r = fl - mu_GP (zero in the
//   padding) and tile (0,0) resets the accumulators of the factorisation.
//   nz (may be null): one byte per tile, in launch order, 1 when the tile as stored holds an entry != 0.0 (NaN included):
//   the exact-zero pattern the factorisation's envelope is computed from (envelope_kernel).  Every lower tile is rewritten
//   by every fill, so the flags need no reset.
//   (Skipping the exponentials that are known to underflow to an exact +0 — a warp-uniform test of a 64-row strip's z
//   range against the column — was measured SLOWER, 71 vs 64 us at N = 6000: with 2.8 km/s pixels and l = 5..7 km/s only
//   a quarter of the strips qualify, and the test's branch keeps the unrolled evaluations from interleaving.)
// ------------------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned nonzero_bits(double v) {
    return ((unsigned)__double2hiint(v) << 1) | (unsigned)__double2loint(v);
}
template <int NCOMP>
__global__ void __launch_bounds__(256) fill_lower_kernel(double* __restrict__ W, int64_t ld, int pad, ZSource zs,
                                                         const double* __restrict__ sigma,
                                                         const double* __restrict__ fl, double mu_GP,
                                                         GpParams gp, double* __restrict__ rvec,
                                                         double* __restrict__ acc, int* __restrict__ info,
                                                         uint8_t* __restrict__ nz) {
    // lower-triangular tile index t -> (bi, bj), bi (bi + 1) / 2 + bj = t
    const int t = blockIdx.x;
    int bi = (int)((sqrtf(8.0f * (float)t + 1.0f) - 1.0f) * 0.5f);
    while ((bi + 1) * (bi + 2) / 2 <= t) ++bi;
    while (bi * (bi + 1) / 2 > t) --bi;
    const int bj = t - bi * (bi + 1) / 2;
    __shared__ double zj[NCOMP][NB];
    __shared__ double etab[64];
    load_exp_table(etab);
    const int tid = threadIdx.x;
    if (tid < NB) {
        int pj = bj * NB + tid;
#pragma unroll
        for (int c = 0; c < NCOMP; ++c) zj[c][tid] = (pj >= pad) ? z_at(zs, c, pj - pad) : 0.0;
        if (bi == bj) rvec[pj] = (pj >= pad) ? __dsub_rn(fl[pj - pad], mu_GP) : 0.0;
    }
    if (bi == 0 && bj == 0 && tid < 8) {
        acc[tid] = 0.0;
        if (tid == 0) info[0] = 0;
    }
    double amp2[NCOMP], p2[NCOMP];
#pragma unroll
    for (int c = 0; c < NCOMP; ++c) gp_coeffs(gp, c, amp2[c], p2[c]);
    const int pi0 = bi * NB + (tid & 63) * 2;
    double zi[NCOMP][2];
#pragma unroll
    for (int e = 0; e < 2; ++e)
#pragma unroll
        for (int c = 0; c < NCOMP; ++c) zi[c][e] = (pi0 + e >= pad) ? z_at(zs, c, pi0 + e - pad) : 0.0;
    double dg[2];
#pragma unroll
    for (int e = 0; e < 2; ++e) {
        double d = amp2[0];
#pragma unroll
        for (int c = 1; c < NCOMP; ++c) d = __dadd_rn(d, amp2[c]);  // pyx:57,:144,:201
        double s = (pi0 + e >= pad) ? sigma[pi0 + e - pad] : 0.0;
        dg[e] = __dadd_rn(d, __dmul_rn(s, s));                        // covariance.py:322
    }
    __syncthreads();
    const int cg = tid >> 6;
    // OR over this thread's entries of their bits below the sign: non-zero unless every entry is +-0 (integer pipe)
    unsigned bits = 0;
    // Interior tiles (strictly below the diagonal, clear of the identity padding) are 95 % of the tiles of a large
    // matrix: no per-entry case analysis there.
    if (bi != bj && (bj > 0 || pad == 0)) {
#pragma unroll 4
        for (int cc = 0; cc < 32; ++cc) {
            const int jl = cc * 4 + cg;
            double v[2];
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                double cov = se_term(amp2[0], p2[0], zi[0][e], zj[0][jl], etab);
#pragma unroll
                for (int c = 1; c < NCOMP; ++c) cov = __dadd_rn(cov, se_term(amp2[c], p2[c], zi[c][e], zj[c][jl], etab));
                v[e] = cov;
            }
            bits |= nonzero_bits(v[0]) | nonzero_bits(v[1]);
            *reinterpret_cast<double2*>(W + pi0 + (int64_t)(bj * NB + jl) * ld) = make_double2(v[0], v[1]);
        }
    } else {
#pragma unroll 4
        for (int cc = 0; cc < 32; ++cc) {
            const int jl = cc * 4 + cg;
            const int pj = bj * NB + jl;
            double v[2];
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const int pi = pi0 + e;
                if (pi < pad || pj < pad) {
                    v[e] = (pi == pj) ? 1.0 : 0.0;
                } else if (pi == pj) {
                    v[e] = dg[e];
                } else {
                    double cov = se_term(amp2[0], p2[0], zi[0][e], zj[0][jl], etab);
#pragma unroll
                    for (int c = 1; c < NCOMP; ++c) cov = __dadd_rn(cov, se_term(amp2[c], p2[c], zi[c][e], zj[c][jl], etab));
                    v[e] = cov;
                }
            }
            bits |= nonzero_bits(v[0]) | nonzero_bits(v[1]);
            *reinterpret_cast<double2*>(W + pi0 + (int64_t)pj * ld) = make_double2(v[0], v[1]);
        }
    }
    if (nz) {
        const int any = __syncthreads_or(bits != 0u);
        if (tid == 0) nz[t] = (uint8_t)any;
    }
}

// ------------------------------------------------------------------------------------------------------
// The envelope of a factorisation, from the fill's exact-zero tile flags (one CTA, right after the fill):
//   f[I]   = first block column J <= I whose tile (I, J) holds a non-zero (I itself when none does)
//   F[I]   = min_{I' >= I} f[I']                 (suffix minimum: row order is only nearly monotone in the shifted z)
//   tend[e] = min{I >= e : F[I] >= e}, or T      (e = 1 .. T; tend[0] = T)
// Row blocks I >= tend[e] are exactly zero in block columns < e, in K and so in L (Cholesky keeps a row's leading
// zeros), so the launches of a panel group ending at panel e stop at row block tend[e] (api.cu launch_factor).
// tend does not decrease with e.  Unsorted data has tend = T everywhere: every launch runs in full.
// F itself is stored too (prof, int[T]): row block I is exactly zero in block columns < F[I], so the update tiles of
// row block I start their k loop at panel F[I] (gemm.cuh SyrkSrc::kfirst).
// ------------------------------------------------------------------------------------------------------
constexpr int ENV_MAX_T = 2048;   // shared-memory suffix minima: matrices up to 262144 rows
__global__ void __launch_bounds__(256) envelope_kernel(const uint8_t* __restrict__ nz, int T, int* __restrict__ tend,
                                                       int* __restrict__ prof) {
    __shared__ int F[ENV_MAX_T];
    pdl_wait();
    const int tid = threadIdx.x;
    for (int I = tid; I < T; I += blockDim.x) {
        const uint8_t* row = nz + (int64_t)I * (I + 1) / 2;
        int J = 0;
        while (J < I && !row[J]) ++J;
        F[I] = J;
    }
    __syncthreads();
    if (tid == 0)
        for (int I = T - 2; I >= 0; --I) F[I] = min(F[I], F[I + 1]);
    __syncthreads();
    for (int I = tid; I < T; I += blockDim.x) prof[I] = F[I];
    for (int e = tid; e <= T; e += blockDim.x) {
        int I = e;
        if (e > 0)
            while (I < T && F[I] < e) ++I;
        tend[e] = (e == 0) ? T : I;
    }
}

// ------------------------------------------------------------------------------------------------------
// Operator-surface fill (fill_V11_f / _f_g / _f_g_h): row-major [N, ld], both triangles + diagonal.
// One CTA per 64x64 tile with I >= J; every off-diagonal pair is evaluated once (i > j, as the reference
// does) and mirrored through shared memory so both stores are coalesced.
// ------------------------------------------------------------------------------------------------------
template <int NCOMP>
__global__ void __launch_bounds__(256) fill_full_kernel(double* __restrict__ mat, int64_t ld, int N, ZSource zs,
                                                        GpParams gp) {
    // lower-triangular tile index t -> (bi, bj), bi (bi + 1) / 2 + bj = t (1-D grid: no empty CTAs)
    const int t = blockIdx.x;
    int bi = (int)((sqrtf(8.0f * (float)t + 1.0f) - 1.0f) * 0.5f);
    while ((bi + 1) * (bi + 2) / 2 <= t) ++bi;
    while (bi * (bi + 1) / 2 > t) --bi;
    const int bj = t - bi * (bi + 1) / 2;
    __shared__ double zi[NCOMP][64], zj[NCOMP][64];
    __shared__ double tile[64][65];
    __shared__ double etab[64];
    load_exp_table(etab);
    const int tid = threadIdx.x;
    if (tid < 64) {
        int i = bi * 64 + tid, j = bj * 64 + tid;
#pragma unroll
        for (int c = 0; c < NCOMP; ++c) {
            zi[c][tid] = (i < N) ? z_at(zs, c, i) : 0.0;
            zj[c][tid] = (j < N) ? z_at(zs, c, j) : 0.0;
        }
    }
    double amp2[NCOMP], p2[NCOMP];
#pragma unroll
    for (int c = 0; c < NCOMP; ++c) gp_coeffs(gp, c, amp2[c], p2[c]);
    double dg = amp2[0];
#pragma unroll
    for (int c = 1; c < NCOMP; ++c) dg = __dadd_rn(dg, amp2[c]);
    __syncthreads();
    const int tx = tid & 63, ty = tid >> 6;
#pragma unroll 4
    for (int r = 0; r < 16; ++r) {
        const int il = ty + 4 * r;
        const int i = bi * 64 + il, j = bj * 64 + tx;
        double cov;
        if (i == j) {
            cov = dg;
        } else {
            // r = z[j] - z[i]; for i < j (diagonal tiles only) this is the negated distance of the mirrored
            // pair, and (p2*r)*r is bit-identical under r -> -r.
            cov = se_term(amp2[0], p2[0], zi[0][il], zj[0][tx], etab);
#pragma unroll
            for (int c = 1; c < NCOMP; ++c) cov = __dadd_rn(cov, se_term(amp2[c], p2[c], zi[c][il], zj[c][tx], etab));
        }
        tile[il][tx] = cov;
        if (i < N && j < N) mat[(int64_t)i * ld + j] = cov;
    }
    if (bi == bj) return;
    __syncthreads();
#pragma unroll 4
    for (int r = 0; r < 16; ++r) {
        const int jl = ty + 4 * r;
        const int i = bi * 64 + tx, j = bj * 64 + jl;
        if (i < N && j < N) mat[(int64_t)j * ld + i] = tile[tx][jl];
    }
}

// fill_V12_f (matrix_functions.pyx:63-94): mat[i,j] = amp2 exp((p2 (cols[j]-rows[i])) (cols[j]-rows[i])).
// NCOMP > 1 sums the per-component cross-covariances (V12_f + V12_g (+ V12_h), covariance.py:167-171).
struct V12Src {
    const double* rows[3];
    const double* cols[3];
};
template <int NCOMP>
__global__ void __launch_bounds__(256) fill_v12_kernel(double* __restrict__ mat, int64_t ld, int M, int N, V12Src src,
                                                       GpParams gp) {
    __shared__ double zr[NCOMP][64];
    __shared__ double etab[64];
    load_exp_table(etab);
    const int tid = threadIdx.x;
    const int i0 = blockIdx.y * 64;
    const int j = blockIdx.x * 64 + (tid & 63);
    double amp2[NCOMP], p2[NCOMP], zc[NCOMP];
#pragma unroll
    for (int c = 0; c < NCOMP; ++c) {
        if (tid < 64) zr[c][tid] = (i0 + tid < M) ? src.rows[c][i0 + tid] : 0.0;
        gp_coeffs(gp, c, amp2[c], p2[c]);
        zc[c] = (j < N) ? src.cols[c][j] : 0.0;
    }
    __syncthreads();
    const int ty = tid >> 6;
#pragma unroll 4
    for (int r = 0; r < 16; ++r) {
        const int il = ty + 4 * r;
        const int i = i0 + il;
        if (i < M && j < N) {
            double cov = se_term(amp2[0], p2[0], zr[0][il], zc[0], etab);
#pragma unroll
            for (int c = 1; c < NCOMP; ++c) cov = __dadd_rn(cov, se_term(amp2[c], p2[c], zr[c][il], zc[c], etab));
            mat[(int64_t)i * ld + j] = cov;
        }
    }
}

// replicate_wls (data.py:40-63)
__global__ void replicate_wls_kernel(double* __restrict__ out, ZSource zs, int64_t N, int ncomp) {
    int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= N) return;
    for (int c = 0; c < ncomp; ++c) out[(int64_t)c * N + k] = z_at(zs, c, k);
}

}  // namespace psoap
