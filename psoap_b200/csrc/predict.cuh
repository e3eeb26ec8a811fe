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

// ---- posterior draws X = delta + L_Sigma Z (psoap_farm_predict_attach_draws) ------------------------------------------
// Philox4x32-10 (Salmon et al., SC'11; the Random123 constants): counter c, key k.
__host__ __device__ __forceinline__ void philox4x32_10(uint32_t (&c)[4], uint32_t k0, uint32_t k1) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint64_t p0 = (uint64_t)0xD2511F53u * c[0], p1 = (uint64_t)0xCD9E8D57u * c[2];
        const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c[1] ^ k0, n2 = (uint32_t)(p0 >> 32) ^ c[3] ^ k1;
        c[0] = n0; c[1] = (uint32_t)p1; c[2] = n2; c[3] = (uint32_t)p0;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
}

// A uniform from two 32-bit outputs: the top 53 bits of (hi << 32 | lo), plus one half, times 2^-53.  Never 0, so the
// logarithm of Box-Muller is finite; the sum rounds to 2^53 for the top 2^11 words, where u = 1 and the pair is 0.
__device__ __forceinline__ double philox_uniform(uint32_t hi, uint32_t lo) {
    const uint64_t v = (((uint64_t)hi << 32) | lo) >> 11;
    return __dmul_rn(__dadd_rn((double)v, 0.5), 0x1p-53);
}

// Standard normals of rows a = 2j and 2j + 1 of draw s for (seed, chunk key, proposal): one Philox block with key
// (seed low, seed high) and counter (j, s, proposal, chunk key), Box-Muller on its two uniforms, the cosine for the
// even row and the sine for the odd one.  Nothing else enters, so a draw's bits do not depend on where or in which
// order it is generated.
__device__ __forceinline__ void normal_pair(uint64_t seed, uint32_t chunk_key, uint32_t proposal, uint32_t s, uint32_t j,
                                            double& z_even, double& z_odd) {
    uint32_t c[4] = {j, s, proposal, chunk_key};
    philox4x32_10(c, (uint32_t)seed, (uint32_t)(seed >> 32));
    const double u1 = philox_uniform(c[0], c[1]), u2 = philox_uniform(c[2], c[3]);
    const double r = sqrt(__dmul_rn(-2.0, log(u1)));
    double sn, cs;
    sincospi(__dmul_rn(2.0, u2), &sn, &cs);
    z_even = __dmul_rn(r, cs);
    z_odd = __dmul_rn(r, sn);
}

// Z[s][a] (row s at out + s ld) for a < M, zero for M <= a < Mrows, s < S.  The seed is *seed_dev when that is not null
// (the prediction graph's own word, set before every replay), else `seed`.  Grid (ceil(Mrows / 256), min(S, 65535)).
__global__ void __launch_bounds__(128) normals_kernel(const uint64_t* __restrict__ seed_dev, uint64_t seed, uint32_t chunk_key,
                                                      uint32_t proposal, int S, int M, int Mrows, double* __restrict__ out,
                                                      int64_t ld) {
    if (seed_dev) seed = *seed_dev;
    const int j = blockIdx.x * blockDim.x + threadIdx.x, a = 2 * j;
    if (a >= Mrows) return;
    for (int s = blockIdx.y; s < S; s += gridDim.y) {
        double z0 = 0.0, z1 = 0.0;
        if (a < M) normal_pair(seed, chunk_key, proposal, (uint32_t)s, (uint32_t)j, z0, z1);
        double* o = out + (int64_t)s * ld;
        o[a] = z0;
        if (a + 1 < Mrows) o[a + 1] = (a + 1 < M) ? z1 : 0.0;
    }
}

// Before the factorisation of Sigma + jitter I in place (the trailing block T of an item, after the read-out): jitter on
// the M live diagonal entries, and the residual [Mp], accumulators and info word of Sigma's own FactorWs zeroed.
__global__ void __launch_bounds__(256) sigma_jitter_kernel(double* __restrict__ T, int64_t ld, int M, int Mp, double jitter,
                                                           double* __restrict__ rvec, double* __restrict__ acc,
                                                           int* __restrict__ info) {
    for (int a = threadIdx.x; a < Mp; a += blockDim.x) {
        if (a < M) T[a + (int64_t)a * ld] = __dadd_rn(T[a + (int64_t)a * ld], jitter);
        rvec[a] = 0.0;
    }
    if (threadIdx.x < 8) acc[threadIdx.x] = 0.0;
    if (threadIdx.x < 2) info[threadIdx.x] = 0;
}

// Block column kb of L into the factored matrix T as its panel finishes (launch_factor's lstore): the diagonal tile from
// Lkk (potrf_diag7's L_kk, column-major [128, 128]) with exact zeros above the diagonal, the R row blocks below it from
// the panel P (rows absolute, leading dimension ldp).  Grid R + 1: CTA 0 the diagonal tile, CTA b row block kb + b.
__global__ void __launch_bounds__(256) store_l_kernel(const double* __restrict__ Lkk, const double* __restrict__ P,
                                                      int64_t ldp, double* __restrict__ T, int64_t ld, int kb) {
    const int I = kb + (int)blockIdx.x;
    const int r = threadIdx.x & (NB - 1);
    double* dst = T + (int64_t)I * NB + r + (int64_t)kb * NB * ld;
    for (int c = threadIdx.x >> 7; c < NB; c += 2) {
        const double v = blockIdx.x == 0 ? (r >= c ? Lkk[r + c * NB] : 0.0) : P[(int64_t)I * NB + r + (int64_t)c * ldp];
        dst[(int64_t)c * ld] = v;
    }
}

// X[s][a] = delta[a] + sum_{k <= a} L[a][k] Z[s][k] for a < M, s < S, row-major at X (row length M); delta[a] = -rtail[a]
// (the carried residual the read-out negates).  L: the lower triangle of T (column-major, ld), read with k <= a, so
// whatever lies above the diagonal is never used; Z: [S][Mp], zero in rows M.. of each draw.  A CTA owns 64 rows a and 64
// draws s; its k loop ends at its diagonal tile.  DMMA m8n8k4 with M <-> s, N <-> a: a thread's two accumulators are
// two consecutive a of one draw.  Warps 2 (s) x 4 (a), each 32 s x 16 a.  Every draw is NaN when the item's sentinel
// fired or either factorisation failed (the data block's info, Sigma's info).
constexpr int DR_T = 64, DR_K = 32, DR_LP = DR_T + 8, DR_ZP = DR_K + 4;
__global__ void __launch_bounds__(256) predict_draws_kernel(const double* __restrict__ T, int64_t ld, int M, int Mp,
                                                            const double* __restrict__ Z, int S,
                                                            const double* __restrict__ rtail, const int* __restrict__ info_data,
                                                            const int* __restrict__ info_sigma, const int* __restrict__ sentinel,
                                                            double* __restrict__ X) {
    __shared__ double sL[DR_K][DR_LP];   // sL[k][a] = L[a0 + a][k0 + k], masked to k <= a
    __shared__ double sZ[DR_T][DR_ZP];   // sZ[s][k] = Z[s0 + s][k0 + k]
    const int a0 = blockIdx.x * DR_T, s0 = blockIdx.y * DR_T;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g4 = lane >> 2, tq = lane & 3;
    const int ws = warp & 1, wa = warp >> 1;
    double acc[4][2][2];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 2; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;
    const int kend = min(a0 + DR_T, Mp);
#pragma unroll 1
    for (int k0 = 0; k0 < kend; k0 += DR_K) {
#pragma unroll
        for (int e = tid; e < DR_K * DR_T; e += 256) {
            const int a = e & (DR_T - 1), k = e / DR_T;
            sL[k][a] = (k0 + k <= a0 + a) ? T[(a0 + a) + (int64_t)(k0 + k) * ld] : 0.0;
        }
#pragma unroll
        for (int e = tid; e < DR_K * DR_T; e += 256) {
            const int k = e & (DR_K - 1), s = e / DR_K;
            sZ[s][k] = (s0 + s < S) ? Z[(k0 + k) + (int64_t)(s0 + s) * Mp] : 0.0;
        }
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < DR_K / 4; ++kk) {
            double fa[4], fb[2];
#pragma unroll
            for (int i = 0; i < 4; ++i) fa[i] = sZ[ws * 32 + i * 8 + g4][kk * 4 + tq];
#pragma unroll
            for (int j = 0; j < 2; ++j) fb[j] = sL[kk * 4 + tq][wa * 16 + j * 8 + g4];
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 2; ++j) dmma_8x8x4(acc[i][j][0], acc[i][j][1], fa[i], fb[j]);
        }
        __syncthreads();
    }
    const bool bad = sentinel[0] != 0 || info_data[0] != 0 || info_sigma[0] != 0;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int s = s0 + ws * 32 + i * 8 + g4;
        if (s >= S) continue;
#pragma unroll
        for (int j = 0; j < 2; ++j)
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const int a = a0 + wa * 16 + j * 8 + 2 * tq + e;
                if (a < M) X[(int64_t)s * M + a] = bad ? CUDART_NAN : __dadd_rn(-rtail[a], acc[i][j][e]);
            }
    }
}

}  // namespace psoap
