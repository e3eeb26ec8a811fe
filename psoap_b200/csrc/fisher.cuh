// fisher.cuh — expected Fisher information of one chunk's Gaussian likelihood in the registered parameters p
// (orbital, then GP):
//
//   F_ab = 1/2 tr(K^-1 dK/dp_a K^-1 dK/dp_b) = 1/2 sum_ij A_a[i,j] A_b[j,i],   A_a = K^-1 D_a,   D_a = dK/dp_a
//
// It runs after the steps of psoap_chunk_lnprob_grad (api.cu), whose outputs it leaves as they are, in the same
// workspace: the identity-bordered elimination has left -K^-1 in the lower triangle of the trailing block, and the data
// block is dead once the gradient contraction has run.
//   1. fisher_mirror_kernel turns the trailing block into the full symmetric K^-1 in place (data order, zero padding).
//   2. Per parameter a: fisher_dk_kernel writes the full symmetric D_a into the data block, and fisher_gemm_kernel
//      forms A_a = K^-1 D_a (gemm_persistent, MODE 0) into a buffer of its own.  D_a is exactly zero wherever every
//      exponential factor of the covariance is (they underflow to +0 beyond about 38.6 length scales): the first
//      launch flags the 128 x 128 tiles that hold a non-zero factor and fisher_krange_kernel turns the flags into the
//      k range of each block column, which the GEMM tiles of that column run over.  The terms left out multiply exact
//      zeros, so A_a is the dense product up to the sign of zeros.
//   3. fisher_pair_kernel contracts each pair of tiles {(I, J), (J, I)} into fixed-order partials, and
//      fisher_reduce_kernel sums them in pair order.  No floating-point atomics: F is bit-reproducible, and symmetric
//      bit for bit (both triangles are written from one value).
#pragma once
#include <math_constants.h>

#include "common.cuh"
#include "fill.cuh"
#include "gemm.cuh"
#include "grad.cuh"

namespace psoap {

constexpr int FISHER_MAXP = 19;    // registered parameters of the largest model (ST3)
constexpr int FISHER_CHUNK = 256;  // tile-pair elements staged per step of fisher_pair_kernel (two columns)
__host__ __device__ constexpr int fisher_pair_smem(int P) { return (2 * FISHER_CHUNK * P + P * P) * 8; }

// -K^-1 in the lower triangle of the trailing block (column-major, leading dimension ld, data order) -> K^-1 in both
// triangles, zero in the padding rows and columns (>= N).  One CTA per 32 x 32 tile pair {(I, J), (J, I)}, I >= J:
// (I, J) is read completely before either tile is written, and only (I, J) is read, so the pairs are independent.
__global__ void __launch_bounds__(256) fisher_mirror_kernel(double* __restrict__ S, int64_t ld, int N) {
    const int t = blockIdx.x;
    int I = (int)((sqrtf(8.0f * (float)t + 1.0f) - 1.0f) * 0.5f);
    while ((I + 1) * (I + 2) / 2 <= t) ++I;
    while (I * (I + 1) / 2 > t) --I;
    const int J = t - I * (I + 1) / 2;
    __shared__ double s[32][33];
    const int r = threadIdx.x & 31, c0 = threadIdx.x >> 5;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int c = c0 + 8 * k;
        const int i = I * 32 + r, j = J * 32 + c;
        s[r][c] = (i < N && j < N && i >= j) ? -S[i + (int64_t)j * ld] : 0.0;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int c = c0 + 8 * k;
        S[(I * 32 + r) + (int64_t)(J * 32 + c) * ld] = (r >= c || I != J) ? s[r][c] : s[c][r];
        if (I != J) S[(J * 32 + r) + (int64_t)(I * 32 + c) * ld] = s[c][r];
    }
}

// D_a = dK/dp_a, both triangles, column-major (leading dimension ld), data order, zero in the padding; one CTA per
// 128 x 128 tile (I = t % Tb, J = t / Tb), thread = 2 consecutive rows, as the fill.  With r = z_j - z_i,
// x = (p2 r) r, e = exp_neg(x), k = amp^2 e (the arithmetic of lnlike_grad_kernel):
//   amp_c:  2 amp_c e_c          l_c:  -2 (k_c x_c) / l_c
//   orbital parameter a:  sum_c ((2 p2_c k_c) r_c) (u_ca[e_j] - u_ca[e_i]),  u_ca[e] = -J_c[e][a] / c_kms
// (dz_c,i/dp_a = u_ca[epoch(i)]).  Swapping i and j negates r and the difference of u and nothing else, so D_a is
// symmetric bit for bit; for gamma (J = 1 at every epoch) the difference, and with it D_a, is exactly zero.
// flags (may be null): one byte per tile, [I][J] row-major, 1 when an exponential factor of a live entry is non-zero
// (the factors, not the sum, so that a tiny amp cannot hide a non-zero dK/damp).
template <int NCOMP>
__global__ void __launch_bounds__(256) fisher_dk_kernel(double* __restrict__ D, int64_t ld, int Tb, int N, ZSource zs,
                                                        GpParams gp, const double* __restrict__ jac, int norb, int a,
                                                        uint8_t* __restrict__ flags) {
    const int I = blockIdx.x % Tb, J = blockIdx.x / Tb;
    const bool orb = a < norb;
    const int ca = orb ? -1 : (a - norb) >> 1;   // the component of a GP parameter
    const bool is_l = !orb && ((a - norb) & 1);
    __shared__ double zj[NCOMP][NB];
    __shared__ double uj[NCOMP][NB];
    __shared__ double etab[64];
    load_exp_table(etab);
    const int tid = threadIdx.x;
    if (tid < NB) {
        const int b = J * NB + tid;
#pragma unroll
        for (int c = 0; c < NCOMP; ++c) {
            zj[c][tid] = (b < N) ? z_at(zs, c, b) : 0.0;
            uj[c][tid] = (orb && b < N) ? -jac[((int64_t)c * zs.n_epochs + zs.epoch[b]) * norb + a] / C_KMS : 0.0;
        }
    }
    double amp2[NCOMP], p2[NCOMP];
#pragma unroll
    for (int c = 0; c < NCOMP; ++c) gp_coeffs(gp, c, amp2[c], p2[c]);
    double amp = 0.0, l = 1.0;
    if (!orb) gp_pick(gp, ca, amp, l);
    const int i0 = I * NB + (tid & 63) * 2;
    double zi[NCOMP][2], ui[NCOMP][2];
#pragma unroll
    for (int e = 0; e < 2; ++e)
#pragma unroll
        for (int c = 0; c < NCOMP; ++c) {
            const int i = i0 + e;
            zi[c][e] = (i < N) ? z_at(zs, c, i) : 0.0;
            ui[c][e] = (orb && i < N) ? -jac[((int64_t)c * zs.n_epochs + zs.epoch[i]) * norb + a] / C_KMS : 0.0;
        }
    __syncthreads();
    const int cg = tid >> 6;
    unsigned bits = 0;
#pragma unroll 2
    for (int cc = 0; cc < 32; ++cc) {
        const int jl = cc * 4 + cg;
        const int j = J * NB + jl;
        double v[2];
#pragma unroll
        for (int e = 0; e < 2; ++e) {
            const bool live = (i0 + e < N) && (j < N);
            double d = 0.0;
#pragma unroll
            for (int c = 0; c < NCOMP; ++c) {
                if (!orb && c != ca && !flags) continue;
                const double r = __dsub_rn(zj[c][jl], zi[c][e]);
                const double x = __dmul_rn(__dmul_rn(p2[c], r), r);
                const double ex = exp_neg(x, etab);
                if (live) bits |= nonzero_bits(ex);
                const double k = __dmul_rn(amp2[c], ex);
                if (orb) {
                    const double du = __dsub_rn(uj[c][jl], ui[c][e]);
                    d = __dadd_rn(d, __dmul_rn(__dmul_rn(__dmul_rn(2.0 * p2[c], k), r), du));
                } else if (c == ca) {
                    d = is_l ? __ddiv_rn(-2.0 * __dmul_rn(k, x), l) : __dmul_rn(2.0 * amp, ex);
                }
            }
            v[e] = live ? d : 0.0;
        }
        *reinterpret_cast<double2*>(D + i0 + (int64_t)j * ld) = make_double2(v[0], v[1]);
    }
    if (flags) {
        const int any = __syncthreads_or(bits != 0u);
        if (tid == 0) flags[(int64_t)I * Tb + J] = (uint8_t)any;
    }
}

// k range of block column J: [krange[2 J], krange[2 J + 1]], the first and last row block I whose tile (I, J) is
// flagged (D_a is symmetric, so these are also the block columns of row block J that can be non-zero).  The diagonal
// tile of a live block always is (exp_neg(0) = 1).
__global__ void __launch_bounds__(256) fisher_krange_kernel(const uint8_t* __restrict__ flags, int Tb,
                                                            int* __restrict__ krange) {
    for (int J = threadIdx.x; J < Tb; J += blockDim.x) {
        int lo = J, hi = J;
        for (int I = 0; I < Tb; ++I)
            if (flags[(int64_t)I * Tb + J]) { lo = min(lo, I); hi = max(hi, I); }
        krange[2 * J] = lo;
        krange[2 * J + 1] = hi;
    }
}

// A_a = S D_a (= S D_a^T, D_a symmetric) over the full Nn x Nn output: 128 x 64 tiles, the row tile fastest (the
// CTAs that run side by side share their D_a columns), k over the rows of block column J = J64 / 2 that can be
// non-zero in D_a.  Map A: S (box SA rows), map B: D_a (box SB rows), both over Nn x Nn blocks of the bordered matrix.
struct FisherSrc {
    const int* krange;
    double* C;      // A_a, column-major [Nn, Nn], leading dimension ldc
    int64_t ldc;
    int Tb;
    template <int SH = 1>
    __device__ __forceinline__ TileDesc tile(int t) const {
        const int I = t % Tb, J64 = t / Tb, J = J64 >> 1;
        const int lo = krange[2 * J], hi = krange[2 * J + 1];
        TileDesc d;
        d.Ai = nullptr; d.lda = 0; d.Bj = nullptr; d.ldb = 0;   // operands come through the tensor maps
        d.kbeg = lo * NB;
        d.KT = (hi - lo + 1) * (NB / BK);
        d.C = C + (int64_t)I * NB + (int64_t)J64 * BJ * ldc;
        d.ldc = ldc;
        d.rowA = I * NB; d.colA0 = 0;
        d.rowB = J64 * BJ; d.colB0 = 0;
        return d;
    }
};

__global__ void __launch_bounds__(256, CTAS_PER_SM)
fisher_gemm_kernel(FisherSrc src, int ntiles, const __grid_constant__ CUtensorMap mapS,
                   const __grid_constant__ CUtensorMap mapD) {
    extern __shared__ __align__(128) double sm[];
    gemm_persistent<0, 1>(src, ntiles, blockIdx.x, gridDim.x, sm, &mapS, &mapD);
}

// index of (a, b), a <= b, in the row-major upper triangle of a P x P matrix
__host__ __device__ __forceinline__ int fisher_tri(int a, int b, int P) { return a * P - a * (a - 1) / 2 + (b - a); }

// Tile pair {(I, J), (J, I)}, I >= J (block t of the lower-triangle enumeration), of the products A_0 .. A_{P-1}
// (column-major [Nn, Nn] each, `stride` doubles apart).  With X_a[e] = A_a[I 128 + i, J 128 + j] and
// Y_a[e] = A_a[J 128 + j, I 128 + i] over the pair's elements e = (i, j), G_ab = sum_e X_a[e] Y_b[e] and
//   part[t][tri(a, b)] = G_ab (I == J)   or   G_ab + G_ba (I > J)        (a <= b)
// so that sum_t part[t][tri(a, b)] = sum_ij A_a[i,j] A_b[j,i].  Elements are staged FISHER_CHUNK at a time as [e][a]
// (a thread's G entries (a, b) read one X and one Y word per term, adjacent b in adjacent banks); each G entry is one
// thread's sum in element order.
__global__ void __launch_bounds__(256) fisher_pair_kernel(const double* __restrict__ A, int64_t stride, int64_t ld,
                                                          int P, double* __restrict__ part) {
    const int t = blockIdx.x;
    int I = (int)((sqrtf(8.0f * (float)t + 1.0f) - 1.0f) * 0.5f);
    while ((I + 1) * (I + 2) / 2 <= t) ++I;
    while (I * (I + 1) / 2 > t) --I;
    const int J = t - I * (I + 1) / 2;
    extern __shared__ __align__(16) double fs[];
    double* X = fs;
    double* Y = X + FISHER_CHUNK * P;
    double* G = Y + FISHER_CHUNK * P;
    const int tid = threadIdx.x;
    const int PP = P * P;
    const int q0 = tid, q1 = tid + 256;   // this thread's G entries (row-major a * P + b)
    const int a0 = q0 / P, b0 = q0 % P, a1 = q1 / P, b1 = q1 % P;
    double g0 = 0.0, g1 = 0.0;
    const int i = tid & (NB - 1), jj = tid >> 7;   // the element this thread stages: row i, column j0 + jj
#pragma unroll 1
    for (int j0 = 0; j0 < NB; j0 += FISHER_CHUNK / NB) {
        const int64_t ox = (int64_t)(I * NB + i) + (int64_t)(J * NB + j0 + jj) * ld;
        const int64_t oy = (int64_t)(J * NB + j0 + jj) + (int64_t)(I * NB + i) * ld;
        for (int a = 0; a < P; ++a) {
            X[tid * P + a] = A[a * stride + ox];
            Y[tid * P + a] = A[a * stride + oy];
        }
        __syncthreads();
        if (q0 < PP) {
#pragma unroll 4
            for (int e = 0; e < FISHER_CHUNK; ++e) g0 = fma(X[e * P + a0], Y[e * P + b0], g0);
        }
        if (q1 < PP) {
#pragma unroll 4
            for (int e = 0; e < FISHER_CHUNK; ++e) g1 = fma(X[e * P + a1], Y[e * P + b1], g1);
        }
        __syncthreads();
    }
    if (q0 < PP) G[q0] = g0;
    if (q1 < PP) G[q1] = g1;
    __syncthreads();
    const int nF = P * (P + 1) / 2;
    for (int q = tid; q < PP; q += 256) {
        const int a = q / P, b = q % P;
        if (a > b) continue;
        part[(int64_t)t * nF + fisher_tri(a, b, P)] = (I == J) ? G[a * P + b] : G[a * P + b] + G[b * P + a];
    }
}

// F (row-major P x P) = 1/2 sum over the tile pairs, in pair order, of the partials; both triangles from one value.
// NaN everywhere when the likelihood is -inf (info != 0, or the sentinel of the orbit / hyper-parameter check fired),
// the words the gradient reads.
__global__ void __launch_bounds__(256) fisher_reduce_kernel(const double* __restrict__ part, int npairs, int P,
                                                            const int* __restrict__ info,
                                                            const int* __restrict__ sentinel, double* __restrict__ F) {
    const int nF = P * (P + 1) / 2;
    const bool bad = grad_flagged(info, sentinel);
    for (int q = threadIdx.x; q < P * P; q += blockDim.x) {
        const int a = q / P, b = q % P;
        if (a > b) continue;
        const int k = fisher_tri(a, b, P);
        double s = 0.0;
        for (int t = 0; t < npairs; ++t) s += part[(int64_t)t * nF + k];
        const double v = bad ? CUDART_NAN : 0.5 * s;
        F[a * P + b] = v;
        F[b * P + a] = v;
    }
}

}  // namespace psoap
