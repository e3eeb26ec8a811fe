// gemm.cuh — persistent DMMA tile GEMM for the panel solve (trsm) and the trailing update (syrk).
//
//   acc[i][j] = sum_k Ai[i,k] * Bj[j,k]      128 x 64 output tile, 256 threads (8 warps, 32 x 32 each)
//
// B200-native structure:
//   * operands are staged by the TMA engine through 2-D tensor maps: per stage of 16 k-columns ONE elected thread
//     issues two cp.async.bulk.tensor.2d (SASS UTMALDG.2D), a box of 132 rows for the 128-row operand and one of
//     68 rows for the 64-row operand, completing on an mbarrier with a transaction count; no thread moves operand
//     data and there is no __syncthreads in the main loop.  The 4 extra rows of a box ARE the shared-memory row
//     padding that makes the m8n8k4 fragment loads bank-conflict free (rows past the matrix edge arrive as zeros).
//   * consumer release goes through a second set of mbarriers ("empty"), so warps drift freely and a stage is
//     refilled two items after it was consumed.
//   * CTAs are persistent (2 per SM) and the TMA pipeline runs ahead ACROSS tiles: the next tile's operands
//     land while the current tile's epilogue (read-modify-write of C in HBM, prefetched into L2 at tile start)
//     is in flight.
//   * math is DMMA.8x8x4 (mma.sync.m8n8k4.f64): FP64 has no tcgen05 kind, DMMA is the FP64 tensor pipe.
//   mma M <-> j, mma N <-> i, so each thread owns two consecutive rows i of a column j: double2 epilogue on the
//   column-major output.
#pragma once
#include <cuda.h>   // CUtensorMap (type only; the encoder is fetched through cudaGetDriverEntryPoint)
#include "common.cuh"

#ifdef __CUDA_ARCH__
#define PSOAP_FSQRT(x) __fsqrt_rn(x)   // FP32: the FP64 pipe belongs to DMMA
#else
#include <cmath>
#define PSOAP_FSQRT(x) sqrtf(x)
#endif

namespace psoap {

constexpr int BI = 128, BJ = 64, BK = 16;
constexpr int GEMM_WARPS = 8;
// Tile shapes.  SH = 1: 128 x 64 output tile (warp tile 32 x 32), the throughput shape of the trailing update.
// SH = 2: 64 x 32 (warp tile 16 x 16), four times as many tiles of a quarter of the work each: the LATENCY shape, for
// the short-K updates on the critical path of a matrix factored on its own (a 128 x 64 x K=128 tile keeps one SM busy
// for 8 us at the FP64 peak; the block column it belongs to has only 2 R of them for the whole GPU).
template <int SH>
struct Shape {
    static constexpr int TI = BI / SH, TJ = BJ / SH;          // tile rows (i), tile columns (j)
    static constexpr int SA = TI + 4, SB = TJ + 4;            // padded operand rows in shared memory (= TMA box rows)
    static constexpr int STAGE = BK * SA + BK * SB;           // doubles per pipeline stage
    // Pipeline depth.  A 64 x 32 tile is short of work per stage (4 DMMAs per warp and k-step), so what bounds it is
    // how many TMA round trips (~1 us each) it has in flight: 8 stages (6 in flight) against 4 (2 in flight).
    static constexpr int NSTAGE = SH == 1 ? 4 : 8;
    static constexpr int SMEM = NSTAGE * STAGE * 8 + 2 * NSTAGE * 8;
    static constexpr int NI = TI / 32, NJ = TJ / 16;          // 8 x 8 atoms per warp along i and j (warps 4 x 2)
};
constexpr int SA = Shape<1>::SA, SB = Shape<1>::SB;
constexpr int STAGE_DOUBLES = Shape<1>::STAGE;
constexpr int GEMM_SMEM = Shape<1>::SMEM;
// syrk3_kernel<1> may carry quarter-tile CTAs (the SH = 2 pipeline) behind its persistent ones: room for either
constexpr int SYRK1_SMEM = Shape<1>::SMEM > Shape<2>::SMEM ? Shape<1>::SMEM : Shape<2>::SMEM;

// 2-D tiled TMA (cp.async.bulk.tensor, SASS UTMALDG): box {rows, 16 k-columns} of a column-major matrix lands as
// [16][rows] in shared memory; with a box of 132 (68) rows that IS the padded, bank-conflict-free stage layout, so a
// whole operand stage is ONE instruction.  c0 = row coordinate, c1 = column coordinate.
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* map, int c0, int c1, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];\n" ::"r"(
            smem_u32(smem_dst)),
        "l"(map), "r"(c0), "r"(c1), "r"(smem_u32(bar))
        : "memory");
}
__device__ __forceinline__ void tma_prefetch_l2(const void* p, uint32_t bytes) {
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;\n" ::"l"(p), "r"(bytes) : "memory");
}

struct TileDesc {
    const double* Ai;  // [128 rows, k] column-major, leading dimension lda
    int64_t lda;
    const double* Bj;  // [64 rows, k]
    int64_t ldb;
    int kbeg, KT;      // k range [kbeg, kbeg + 16 KT), KT >= 1
    double* C;         // [128, 64] column-major output tile
    int64_t ldc;
    int rowA, rowB;    // tensor-map path: first row of the operands in their maps
    int colA0, colB0;  //                  column of k = 0 in their maps
};

// trsm tiles: rows below panel kb.  tile t -> row tile I = kb+1 + t/2, column half jh = t%2:
//   P[I*128 + :, jh*64 + :] = W[I*128 + :, kb*128 + (0 .. (jh+1)*64)] * Linv[jh*64 + :, same]^T
struct TrsmSrc {
    const double* W;
    int64_t ld;
    int kb, kbeg;
    const double* Linv;
    double* P;
    int64_t ldp;
    const int* tend = nullptr;   // envelope (may be null): row blocks from tend[tend_at] on are skipped (see row_limit)
    int tend_at = 0;
    template <int SH = 1>
    __device__ __forceinline__ TileDesc tile(int t) const {
        const int I = kb + 1 + (t >> 1), jh = t & 1;
        const int kend = (jh + 1) * BJ;
        const int kb0 = min(kbeg, kend - BK);  // keep KT >= 1 (leading identity-padding columns only add zeros)
        TileDesc d;
        d.Ai = W + (int64_t)I * NB + (int64_t)kb * NB * ld;
        d.lda = ld;
        d.Bj = Linv + jh * BJ;
        d.ldb = NB;
        d.kbeg = kb0;
        d.KT = (kend - kb0) / BK;
        d.C = P + (int64_t)I * NB + (int64_t)jh * BJ * ldp;
        d.ldc = ldp;
        d.rowA = I * NB; d.colA0 = kb * NB;   // map A: W
        d.rowB = jh * BJ; d.colB0 = 0;        // map B: Linv
        return d;
    }
};

// syrk tiles: W[I, J] -= P_I P_J^T over the row tiles I = row0 + r, r in [0, R), with P the panel buffer
// [Nt, 128 G] (the G adjacent 128-wide panels of a group; k range [kbeg, kend), kend a multiple of 128).  Row r owns the 128 x 64
// tiles jrel in [0, 2r+2), J64 = 2 row0 + jrel.
//   part 0: all of them
//   part 1: jrel < ncol1 (ncol1 = 2 per panel of the next group: its block columns, for look-ahead)
//   part 2: jrel >= ncol1
struct SyrkSrc {
    double* W;
    int64_t ld;
    int row0, kbeg, kend;   // row0 in units of the tile rows (128, or 64 for the small shape)
    int res_row0;           // first 128-row block of the residual update
    const double* P;
    int64_t ldp;
    int part, ncol1;
    const int* tend = nullptr;   // envelope (may be null): row blocks from tend[tend_at] on are skipped (see row_limit)
    int tend_at = 0;
    static constexpr bool PREFETCH_C = true;   // the next tile's C lines are pulled towards L2 (gemm_persistent)
    // tile index -> (row r, 64-column tile jrel); host-callable so the CPU tests can check the coverage
    __host__ __device__ __forceinline__ void decode(int t, int& r, int& jrel) const {
        if (part == 0) {
            r = (int)((PSOAP_FSQRT(4.0f * (float)t + 1.0f) - 1.0f) * 0.5f);
            while ((r + 1) * (r + 2) <= t) ++r;
            while (r * (r + 1) > t) --r;
            jrel = t - r * (r + 1);
        } else if (part == 1) {
            // rows r < h = ncol1/2 are still triangular (2r+2 tiles), rows r >= h have ncol1 tiles each
            const int h = ncol1 >> 1, tri = h * (h + 1);
            if (t < tri) {
                r = (int)((PSOAP_FSQRT(4.0f * (float)t + 1.0f) - 1.0f) * 0.5f);
                while ((r + 1) * (r + 2) <= t) ++r;
                while (r * (r + 1) > t) --r;
                jrel = t - r * (r + 1);
            } else {
                r = h + (t - tri) / ncol1;
                jrel = (t - tri) % ncol1;
            }
        } else {
            int v = (int)((PSOAP_FSQRT(4.0f * (float)t + 1.0f) + 1.0f) * 0.5f);
            while ((v + 1) * v <= t) ++v;
            while (v * (v - 1) > t) --v;
            jrel = ncol1 + t - v * (v - 1);
            r = v + (ncol1 >> 1) - 1;
        }
    }
    // SH = 2: the same enumeration in units of 64-row / 32-column tiles (row0, R, ncol1 are then given in those units;
    // a row tile still owns 2 r + 2 column tiles because TI = 2 TJ in both shapes)
    template <int SH = 1>
    __device__ __forceinline__ TileDesc tile(int t) const {
        constexpr int TI = Shape<SH>::TI, TJ = Shape<SH>::TJ;
        int r, jrel;
        decode(t, r, jrel);
        const int I = row0 + r;
        const int J = 2 * row0 + jrel;
        TileDesc d;
        d.Ai = P + (int64_t)I * TI;
        d.lda = ldp;
        d.Bj = P + (int64_t)J * TJ;
        d.ldb = ldp;
        d.kbeg = kbeg;
        d.KT = (kend - kbeg) / BK;
        d.C = W + (int64_t)I * TI + (int64_t)J * TJ * ld;
        d.ldc = ld;
        d.rowA = I * TI; d.rowB = J * TJ; d.colA0 = d.colB0 = 0;   // both operands: the group buffer's map
        return d;
    }
};

// The last, partial round of a persistent launch as QUARTER tiles (64 x 32, the SH = 2 shape): quarter t of the tail
// belongs to the 128 x 64 tile first + t / 4.  Each quarter is one CTA behind the persistent ones in the same grid, so
// the hardware hands them to SM slots as these free up (see syrk3_kernel).  Same k order per entry: same bits.
struct SyrkTailSrc {
    SyrkSrc base;
    int first;
    static constexpr bool PREFETCH_C = false;   // each quarter CTA reads its one C tile without an L2 prefetch
    template <int SH = 2>
    __device__ __forceinline__ TileDesc tile(int t) const {
        TileDesc d = base.template tile<1>(first + (t >> 2));
        const int qi = t & 1, qj = (t >> 1) & 1;
        d.Ai += qi * Shape<2>::TI; d.rowA += qi * Shape<2>::TI;
        d.Bj += qj * Shape<2>::TJ; d.rowB += qj * Shape<2>::TJ;
        d.C += qi * Shape<2>::TI + (int64_t)qj * Shape<2>::TJ * d.ldc;
        return d;
    }
};

// number of tiles of a syrk launch over R row tiles
__host__ __device__ inline int syrk_ntiles(int R, int part, int ncol1) {
    const int h = ncol1 >> 1;
    if (part == 0) return R * (R + 1);
    if (part == 1) return R <= h ? R * (R + 1) : h * (h + 1) + (R - h) * ncol1;
    return R > h ? (R - h) * (R - h + 1) : 0;
}

// Row blocks [row0, row0 + R) of a launch over R row blocks that lie inside the envelope: R, or fewer when the
// envelope (written on the device after the fill, api.cu launch_chunk) says the rows from tend[tend_at] on are exactly
// zero in every panel of the group.  Read after pdl_wait().  The grid and the host's launch plan stay sized for R.
__device__ __forceinline__ int row_limit(const int* tend, int tend_at, int row0, int R) {
    return tend ? max(0, min(R, tend[tend_at] - row0)) : R;
}

__device__ __forceinline__ double flip_sign(double x) {  // integer pipe, keeps the FP64 pipe for DMMA
    return __hiloint2double(__double2hiint(x) ^ 0x80000000, __double2loint(x));
}

// MODE 0: C = acc, 1: C -= acc.  Operands staged by 2-D tensor-map TMA: one elected thread, two instructions per stage.
template <int MODE, int SH, class Src>
__device__ __forceinline__ void gemm_persistent(const Src& src, int ntiles, int first_tile, int tile_stride, double* sm,
                                                const CUtensorMap* mapA, const CUtensorMap* mapB) {
    using TS = Shape<SH>;
    constexpr int SA = TS::SA, SB = TS::SB, STAGE_DOUBLES = TS::STAGE, NI = TS::NI, NJ = TS::NJ, STAGES = TS::NSTAGE;
    const int tid = threadIdx.x;
    const int warp = tid >> 5, lane = tid & 31;
    const int g4 = lane >> 2, tq = lane & 3;
    const int wi = warp & 3, wj = warp >> 2;
    uint64_t* full = reinterpret_cast<uint64_t*>(sm + STAGES * STAGE_DOUBLES);
    uint64_t* empty = full + STAGES;
    if (tid == 0) {
#pragma unroll
        for (int s = 0; s < STAGES; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], GEMM_WARPS);
        }
        mbar_fence_init();
    }
    __syncthreads();

    // ---- producer cursor: which (tile, k-chunk) the next issued stage belongs to.  The stage consumed at
    // item g is refilled at item g + 2 (LAG), so the producing lane practically never spins on the slowest warp.
#ifndef PSOAP_LAG
#define PSOAP_LAG 2
#endif
    constexpr int LAG = PSOAP_LAG;
    int p_tile = first_tile, p_kt = 0, produced = 0;
    bool p_valid = p_tile < ntiles;
    TileDesc pd;
    if (p_valid) pd = src.template tile<SH>(p_tile);
    auto produce = [&]() {
        const int s = produced % STAGES;
        if (tid == 0) {
            if (produced >= STAGES) mbar_wait(&empty[s], ((produced / STAGES) - 1) & 1);
            double* sA = sm + s * STAGE_DOUBLES;
            double* sB = sA + BK * SA;
            const int k0 = pd.kbeg + p_kt * BK;
            mbar_arrive_expect_tx(&full[s], STAGE_DOUBLES * 8);
            tma_load_2d(sA, mapA, pd.rowA, pd.colA0 + k0, &full[s]);
            tma_load_2d(sB, mapB, pd.rowB, pd.colB0 + k0, &full[s]);
        }
        ++produced;
        if (++p_kt == pd.KT) {
            p_kt = 0;
            p_tile += tile_stride;
            p_valid = p_tile < ntiles;
            if (p_valid) pd = src.template tile<SH>(p_tile);
        }
    };
#pragma unroll 1
    for (int s = 0; s < STAGES - LAG && p_valid; ++s) produce();

    const int64_t coff0 = (wi * 8 * NI + tq * 2);
    const int joff0 = wj * 8 * NJ + g4;
    // pull a tile's C lines (TI rows x TJ columns, read-modify-written by this CTA) towards L2 ahead of use: one TMA
    // bulk prefetch per column, where the tile source asks for it
    auto prefetch_c = [&](const TileDesc& t) {
        if constexpr (MODE == 1) {
            if constexpr (Src::PREFETCH_C)
                if (lane < TS::TJ / 8) tma_prefetch_l2(t.C + (int64_t)(warp * (TS::TJ / 8) + lane) * t.ldc, TS::TI * 8);
        }
    };
    if (MODE == 1 && first_tile < ntiles) prefetch_c(src.template tile<SH>(first_tile));

    int g = 0;  // consumed items
#pragma unroll 1
    for (int tile = first_tile; tile < ntiles; tile += tile_stride) {
        const TileDesc td = src.template tile<SH>(tile);
        double* cbase = td.C + coff0 + (int64_t)joff0 * td.ldc;
        double acc[NJ][NI][2];
        // trailing update: a warp whose sub-tile lies strictly above the diagonal (6 of the 16 warps of a diagonal
        // tile pair) has nothing to do: the factorisation reads the lower triangle only.  It keeps the pipeline's
        // barrier protocol and leaves the tensor pipe to the other warps of the SM.
        const bool idle = (MODE == 1) && (td.rowA + wi * 8 * NI + 8 * NI - 1 < td.rowB + wj * 8 * NJ);
        if (MODE == 1 && idle) {
            if (tile + tile_stride < ntiles) prefetch_c(src.template tile<SH>(tile + tile_stride));
        } else if (MODE == 1) {
            // C is read straight into the accumulators at tile start (its lines were prefetched into L2 one tile
            // ago); the DMMAs then run on -C so that the epilogue is a sign flip and a store, with no load latency.
#pragma unroll
            for (int mj = 0; mj < NJ; ++mj)
#pragma unroll
                for (int ni = 0; ni < NI; ++ni) {
                    const double2 v = *reinterpret_cast<const double2*>(cbase + ni * 8 + (int64_t)(mj * 8) * td.ldc);
                    acc[mj][ni][0] = v.x;
                    acc[mj][ni][1] = v.y;
                }
            if (tile + tile_stride < ntiles) prefetch_c(src.template tile<SH>(tile + tile_stride));  // while this tile computes
        } else {
#pragma unroll
            for (int a = 0; a < NJ; ++a)
#pragma unroll
                for (int b = 0; b < NI; ++b) acc[a][b][0] = acc[a][b][1] = 0.0;
        }

#pragma unroll 1
        for (int kt = 0; kt < td.KT; ++kt, ++g) {
            if (p_valid) produce();  // refills the stage consumed LAG items ago
            const int s = g % STAGES;
            mbar_wait(&full[s], (g / STAGES) & 1);
            if (MODE == 1 && kt == 0 && !idle) {
#pragma unroll
                for (int mj = 0; mj < NJ; ++mj)
#pragma unroll
                    for (int ni = 0; ni < NI; ++ni) {
                        acc[mj][ni][0] = flip_sign(acc[mj][ni][0]);
                        acc[mj][ni][1] = flip_sign(acc[mj][ni][1]);
                    }
            }
            const double* sA = sm + s * STAGE_DOUBLES;
            const double* sB = sA + BK * SA;
            if (!idle) {
#pragma unroll
            for (int kk = 0; kk < BK / 4; ++kk) {
                double a[NJ], b[NI];
#pragma unroll
                for (int mj = 0; mj < NJ; ++mj) a[mj] = sB[(kk * 4 + tq) * SB + wj * 8 * NJ + mj * 8 + g4];
#pragma unroll
                for (int ni = 0; ni < NI; ++ni) b[ni] = sA[(kk * 4 + tq) * SA + wi * 8 * NI + ni * 8 + g4];
#pragma unroll
                for (int mj = 0; mj < NJ; ++mj)
#pragma unroll
                    for (int ni = 0; ni < NI; ++ni) dmma_8x8x4(acc[mj][ni][0], acc[mj][ni][1], a[mj], b[ni]);
            }
            }
            // Release the stage only after this warp's fragment loads have RETURNED: ptxas is free to hoist the
            // arrive above the trailing DMMAs (it has no register dependence on them), and an mbarrier arrive
            // is not ordered behind ld.shared still queued in the LSU.  fence.acq_rel.cta (MEMBAR.CTA) drains them.
            asm volatile("fence.acq_rel.cta;\n" ::: "memory");
            __syncwarp();
            if (lane == 0) mbar_arrive(&empty[s]);
        }

        if (!idle) {
#pragma unroll
        for (int mj = 0; mj < NJ; ++mj)
#pragma unroll
            for (int ni = 0; ni < NI; ++ni) {
                double2 v;
                if (MODE == 1) {
                    v.x = flip_sign(acc[mj][ni][0]);
                    v.y = flip_sign(acc[mj][ni][1]);
                } else {
                    v = make_double2(acc[mj][ni][0], acc[mj][ni][1]);
                }
                *reinterpret_cast<double2*>(cbase + ni * 8 + (int64_t)(mj * 8) * td.ldc) = v;
            }
        }
    }
}

// Persistent launch geometry: `nctas` CTAs walk the tiles round-robin, CTAS_PER_SM of them resident per SM (the
// kernels are compiled for that occupancy; persistent_ctas and syrk_split in api.cu fill that many slots per SM).
constexpr int CTAS_PER_SM = 2;
__global__ void __launch_bounds__(256, CTAS_PER_SM)
trsm3_kernel(TrsmSrc src, int ntiles, const __grid_constant__ CUtensorMap mapW, const __grid_constant__ CUtensorMap mapLinv) {
    extern __shared__ __align__(128) double sm[];
    TL_IN();
    pdl_trigger();   // small grid: let the trailing update become resident behind it
    pdl_wait();
    TL_GO(6);
    ntiles = 2 * row_limit(src.tend, src.tend_at, src.kb + 1, ntiles >> 1);
    gemm_persistent<0, 1>(src, ntiles, blockIdx.x, gridDim.x, sm, &mapW, &mapLinv);
    TL_OUT();
}

// residual block: r_I -= P_I[:, res_col0 .. res_col0+128) y for row tile I = row0 + block (deterministic two-half sum)
__device__ __forceinline__ void syrk_residual_block(const SyrkSrc& src, const double* __restrict__ yk,
                                                    double* __restrict__ rvec, int res_col0, double* sm) {
    const int I = src.res_row0 + (int)blockIdx.x;
    const int tid = threadIdx.x;
    const int row = tid & (NB - 1), half = tid >> 7;
    const double* p = src.P + (int64_t)I * NB + row + (int64_t)(res_col0 + half * 64) * src.ldp;
    double s = 0.0;
#pragma unroll 8
    for (int c = 0; c < 64; ++c) s = fma(p[(int64_t)c * src.ldp], yk[half * 64 + c], s);
    sm[tid] = s;
    __syncthreads();
    if (half == 0) rvec[I * NB + row] -= (sm[row] + sm[NB + row]);
}

// Blocks [0, nres) update the residual r_I -= P_I[:, res_col0 .. res_col0+128) y for row tile I = row0 + block
// (deterministic two-half sum); they come FIRST so they are not left waiting for a slot behind the persistent
// tile workers, blocks [nres, nres + nctas), which walk tiles [0, ntiles) round-robin.  Blocks behind those (SH = 1
// only) each take ONE quarter of the tiles from `ntiles` on: the partial last round of a persistent launch, cut into
// 64 x 32 pieces that the block scheduler deals out as the persistent CTAs retire (m = 4096, K = 512: 1056 tiles on
// 296 slots are 3 rounds + 168 tiles; as a 4th round those keep 57 % of the slots busy for a whole tile time).
template <int SH>
__global__ void __launch_bounds__(256, CTAS_PER_SM)
syrk3_kernel(SyrkSrc src, int ntiles, int nctas, int nres, const double* __restrict__ yk, double* __restrict__ rvec,
             int res_col0, const __grid_constant__ CUtensorMap mapPa, const __grid_constant__ CUtensorMap mapPb,
             const __grid_constant__ CUtensorMap mapQa, const __grid_constant__ CUtensorMap mapQb) {
    extern __shared__ __align__(128) double sm[];
    TL_IN();
    pdl_wait();
    TL_GO(SH == 1 ? (src.part == 1 ? 8 : 3) : 4);
    const int b = (int)blockIdx.x - nres;
    // tiles of the rows inside the envelope: a prefix of the launch's tile order (every part enumerates row by row)
    int ntot = 1 << 30;
    if (src.tend) {
        const int R = row_limit(src.tend, src.tend_at, src.res_row0, 1 << 30);
        ntot = syrk_ntiles(SH * R, src.part, src.ncol1);
        nres = min(nres, R);
    }
    if (b < 0) {
        if ((int)blockIdx.x < nres) syrk_residual_block(src, yk, rvec, res_col0, sm);
    } else if (b < nctas) {
        // same buffer, two boxes: TI + 4 rows for the i operand, TJ + 4 rows for the j operand
        gemm_persistent<1, SH>(src, min(ntiles, ntot), b, nctas, sm, &mapPa, &mapPb);
    } else if constexpr (SH == 1) {
        SyrkTailSrc tail;
        tail.base = src; tail.first = ntiles;
        const int q = b - nctas;
        if (ntiles + (q >> 2) < ntot) gemm_persistent<1, 2>(tail, q + 1, q, 1 << 30, sm, &mapQa, &mapQb);
    }
    TL_OUT();
}


}  // namespace psoap
