// api.cu — host orchestration and the C ABI (include/psoap_b200.h) of the sm_100a PSOAP likelihood path.
#include <cudaTypedefs.h>
#include <math_constants.h>

#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <mutex>
#include <numeric>
#include <string>
#include <vector>

#include "../../include/psoap_b200.h"
#include "chain.cuh"
#include "chol.cuh"
#include "common.cuh"
#include "fill.cuh"
#include "fisher.cuh"
#include "gemm.cuh"
#include "grad.cuh"
#include "orbit.cuh"
#include "predict.cuh"

using namespace psoap;

namespace {

thread_local std::string g_err;
std::atomic<int64_t> g_launches{0};

int fail(int code, const std::string& msg) {
    g_err = msg;
    return code;
}
#define CUDA_TRY(expr)                                                                           \
    do {                                                                                         \
        cudaError_t e_ = (expr);                                                                 \
        if (e_ != cudaSuccess)                                                                   \
            return fail(PSOAP_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(e_));     \
    } while (0)
#define LAUNCH_CHECK()                                                                           \
    do {                                                                                         \
        ++g_launches;                                                                            \
        cudaError_t e_ = cudaGetLastError();                                                     \
        if (e_ != cudaSuccess) return fail(PSOAP_ERR_CUDA, std::string("launch: ") + cudaGetErrorString(e_)); \
    } while (0)

inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }
inline int64_t padded_dim(int64_t n) { return (n + NB - 1) / NB * NB; }

// ---- 2-D tensor maps for the TMA operand loads (driver entry point fetched at run time: no -lcuda) ----------
PFN_cuTensorMapEncodeTiled g_encode_tiled = nullptr;

// column-major FP64 matrix [rows, cols] with leading dimension ld; box = {box_rows, 16 columns}
int make_tensor_map(CUtensorMap* m, const double* base, uint64_t rows, uint64_t cols, uint64_t ld, uint32_t box_rows,
                    uint32_t box_cols = BK) {
    const cuuint64_t gdim[2] = {rows, cols};
    const cuuint64_t gstride[1] = {ld * 8};
    const cuuint32_t box[2] = {box_rows, box_cols};
    const cuuint32_t estr[2] = {1, 1};
    CUresult r = g_encode_tiled(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, (void*)base, gdim, gstride, box, estr,
                                CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                                CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(PSOAP_ERR_CUDA, "cuTensorMapEncodeTiled failed (" + std::to_string((int)r) + ")");
    return PSOAP_OK;
}

std::once_flag g_attr_once;
int g_attr_status = 0;
int g_attr_device = 0;
int g_num_sms = 148;
int g_yield_lookahead = 0;  // PSOAP_YIELD_LOOKAHEAD=1|2: how the bulk update shares the SMs with the links under look-ahead (see the syrk launch); 0 = by size
// Chain links (diagonal block + panel solve): 7 = potrf_diag7 + trsm7 (chain.cuh: blocked factorisation with one chain
// warp, blocked substitution), 3 = potrf_diag3 + trsm3 (explicit 128 x 128 inverse, GEMM panel solve).  7 is the faster
// chain for a matrix factored on its own (N = 2000: 0.88 vs 1.22 ms, N = 4000: 2.11 vs 2.74 ms); inside the graph farm,
// where chain latency is hidden by the other chunks and SM-time is what counts, 3 wins (trsm7 keeps a whole SM per
// 32-row tile: see farm_issue).  PSOAP_POTRF sets this default of the direct API.
int g_potrf_version = 7;
// PSOAP_TAIL=1: the partial last round of a trailing update is dealt out as quarter tiles (syrk_split).  Measured on
// a B200: the kernel ALONE gains (m = 4096, K = 512: 29.4 -> 31.7 TFLOP/s, m = 8192: 33.0 -> 33.9), every path that
// ships loses, because there the partial round is already covered by other work: the 256-chunk farm 217.7 -> 224.1 ms
// (the other branches' kernels), a lone N = 6000 matrix 3.71 -> 3.74 ms (the look-ahead's next panels).  Off.
int g_tail_split = 0;
int g_lookahead = 1;   // direct API: next group's head on a high-priority side stream
int g_pdl = 256;       // direct issue: grids up to this many CTAs are launched with programmatic stream serialization
                       // (64 -> 256 with the 32-row panel-solve tiles and 64 x 32 update tiles: N = 2000 0.78 -> 0.72 ms)
int g_group = 0;  // 0: automatic (see launch_factor); PSOAP_GROUP=2|4|8 forces it
inline int persistent_ctas(int ntiles) { return std::max(1, std::min(ntiles, CTAS_PER_SM * g_num_sms)); }
// How a trailing update of `ntiles` 128 x 64 tiles is dealt out: `nmain` tiles to `nctas` CTAs (persistent round-robin,
// or one tile each when `one_per_cta`), and the partial last round, `ntiles - nmain` tiles, as 4 quarter-tile CTAs each
// when that is shorter than one more whole-tile round (3 quarter rounds or fewer).
struct SyrkSplit { int nmain, nctas, nquarters; };
inline SyrkSplit syrk_split(int ntiles, bool one_per_cta, bool allow_tail) {
    const int slots = CTAS_PER_SM * g_num_sms;
    SyrkSplit sp{ntiles, 0, 0};
    const int rem = ntiles % slots;
    if (allow_tail && rem > 0 && 4 * rem <= 3 * slots) { sp.nmain = ntiles - rem; sp.nquarters = 4 * rem; }
    sp.nctas = one_per_cta ? sp.nmain : std::min(sp.nmain, slots);
    return sp;
}
int set_kernel_attributes() {
    std::call_once(g_attr_once, [] {
        cudaError_t e = cudaFuncSetAttribute(potrf_diag3_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, POTRF_SMEM);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(potrf_diag7_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, POTRF7_SMEM);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(trsm7_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, TRSM7_SMEM);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(trsm3_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, GEMM_SMEM);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(syrk3_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, SYRK1_SMEM);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(syrk3_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, Shape<2>::SMEM);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(fisher_gemm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, GEMM_SMEM);
        if (e == cudaSuccess)
            e = cudaFuncSetAttribute(fisher_pair_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, fisher_pair_smem(FISHER_MAXP));
        // every kernel of the chain asks for the same (maximal) shared-memory carve-out: CTAs of kernels with different
        // carve-outs do not share an SM, and the links are meant to run beside the trailing update's CTAs
        if (e == cudaSuccess) e = cudaFuncSetAttribute(potrf_diag3_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(potrf_diag7_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(trsm7_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(trsm3_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(syrk3_kernel<1>, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(syrk3_kernel<2>, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
        int dev = 0;
        if (e == cudaSuccess) e = cudaGetDevice(&dev);
        if (e == cudaSuccess) e = cudaDeviceGetAttribute(&g_num_sms, cudaDevAttrMultiProcessorCount, dev);
        g_attr_device = dev;
        g_attr_status = (int)e;
        if (const char* c = getenv("PSOAP_YIELD_LOOKAHEAD")) g_yield_lookahead = (atoi(c) == 1 || atoi(c) == 2) ? atoi(c) : 0;
        if (const char* c = getenv("PSOAP_POTRF")) g_potrf_version = (atoi(c) == 7) ? 7 : 3;
        if (const char* c = getenv("PSOAP_TAIL")) g_tail_split = atoi(c);
        if (e == cudaSuccess) {
            void* fn = nullptr;
            cudaDriverEntryPointQueryResult qres;
            if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) == cudaSuccess &&
                qres == cudaDriverEntryPointSuccess && fn)
                g_encode_tiled = (PFN_cuTensorMapEncodeTiled)fn;
            else
                e = cudaErrorNotSupported;   // the tensor-map TMA path is the only operand staging there is
        }
        if (const char* c = getenv("PSOAP_LOOKAHEAD")) g_lookahead = atoi(c);
        if (const char* c = getenv("PSOAP_PDL")) g_pdl = atoi(c);
        if (const char* c = getenv("PSOAP_GROUP")) g_group = (atoi(c) >= 8) ? 8 : (atoi(c) >= 4) ? 4 : (atoi(c) >= 2 ? 2 : (atoi(c) == 1 ? 1 : 0));
    });
    if (g_attr_status != 0)
        return fail(PSOAP_ERR_CUDA, std::string("cudaFuncSetAttribute: ") + cudaGetErrorString((cudaError_t)g_attr_status));
    // Kernel attributes, the SM count, the side lane of the direct API and the host-entry staging buffer belong to the
    // device that was current at the first call: one process per GPU (how the path is deployed).  A second device in
    // the same process is refused here rather than failing later with invalid-resource-handle launches.
    int dev = -1;
    if (cudaGetDevice(&dev) != cudaSuccess || dev != g_attr_device)
        return fail(PSOAP_ERR_ARG, "psoap_b200 is bound to CUDA device " + std::to_string(g_attr_device) +
                                       " for the lifetime of the process (one process per GPU); the current device is " +
                                       std::to_string(dev));
    return PSOAP_OK;
}

// Device scratch of one factorisation: W [Nt x Nt] (Nt = padded total dimension), two panel buffers,
// L_kk^-1, residual, y, accumulators, info, the fill's exact-zero tile flags and the envelope computed from them.
constexpr int MAX_GROUP = 8;  // panels per trailing update (rank 128 * G)
struct FactorWs {
    double* W;
    double* P[2];   // two group buffers, each column-major [Nt, 128 * MAX_GROUP] (the adjacent panels of a group)
    double* Linv;   // potrf_diag3: L_kk^-1;  potrf_diag7: L_kk
    double* Xd;     // potrf_diag7: inverses of the four 32 x 32 diagonal sub-blocks of L_kk
    double* rvec;
    double* y;
    double* acc;
    int* info;
    uint8_t* nz;    // fill_lower_kernel: one byte per lower tile, T (T + 1) / 2 (T = Nt / 128)
    int* tend;      // envelope_kernel: int[T + 1], tend[e] = first row block of the envelope of panels [0, e)
    int64_t Nt;
};

size_t factor_ws_bytes(int64_t Nt) {
    size_t b = 0;
    b += align_up((size_t)Nt * Nt * 8, 256);
    b += 2 * align_up((size_t)Nt * MAX_GROUP * NB * 8, 256);
    b += align_up((size_t)NB * NB * 8, 256);
    b += align_up((size_t)4 * XD_BLOCK * 8, 256);
    b += 2 * align_up((size_t)Nt * 8, 256);
    b += align_up(8 * 8, 256);
    b += align_up(2 * 4, 256);
    const int64_t T = Nt / NB;
    b += align_up((size_t)(T * (T + 1) / 2), 256);
    b += align_up((size_t)(T + 1) * 4, 256);
    return b;
}

void carve_factor_ws(char* base, int64_t Nt, FactorWs* ws, bool with_W) {
    char* p = base;
    auto take = [&](size_t bytes) { char* r = p; p += align_up(bytes, 256); return r; };
    ws->Nt = Nt;
    ws->W = with_W ? (double*)take((size_t)Nt * Nt * 8) : nullptr;
    ws->P[0] = (double*)take((size_t)Nt * MAX_GROUP * NB * 8);
    ws->P[1] = (double*)take((size_t)Nt * MAX_GROUP * NB * 8);
    ws->Linv = (double*)take((size_t)NB * NB * 8);
    ws->Xd = (double*)take((size_t)4 * XD_BLOCK * 8);
    ws->rvec = (double*)take((size_t)Nt * 8);
    ws->y = (double*)take((size_t)Nt * 8);
    ws->acc = (double*)take(8 * 8);
    ws->info = (int*)take(2 * 4);
    const int64_t T = Nt / NB;
    ws->nz = (uint8_t*)take((size_t)(T * (T + 1) / 2));
    ws->tend = (int*)take((size_t)(T + 1) * 4);
}

// Streams of one factorisation pipeline: the caller's stream plus a high-priority side stream on which the next
// panel is factored while the bulk of the current trailing update runs (look-ahead).
struct Lanes {
    cudaStream_t main;
    cudaStream_t side;   // may be null: no look-ahead
    cudaEvent_t e1, e2;
    int group = 0;       // panels per trailing update (2 or 4); 0 = choose from the problem size
    int chain = 0;       // chain links: 3 or 7; 0 = g_potrf_version
    int pdl = 0;         // grids of at most this many CTAs are launched with programmatic stream serialization (0: none)
};

// Launch with or without the programmatic-stream-serialization attribute: with it the kernel may become resident
// while its predecessor in the stream still runs, and waits in pdl_wait() (common.cuh).  Only SMALL grids are
// pre-staged: a waiting CTA holds its SM slot, which is free when the chain is the only work (small matrices, the
// tail of a large one) and costly while a big trailing update wants every slot.
template <typename... KArgs, typename... Args>
cudaError_t launch_k(void (*kernel)(KArgs...), dim3 grid, unsigned block, size_t smem, cudaStream_t s, int pdl_max,
                     Args&&... args) {
    const bool pdl = (int)(grid.x * grid.y * grid.z) <= pdl_max;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = dim3(block); cfg.dynamicSmemBytes = smem; cfg.stream = s;
    cudaLaunchAttribute at[1];
    int n = 0;
    if (pdl) {
        at[n].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        at[n].val.programmaticStreamSerializationAllowed = 1;
        ++n;
    }
    cfg.attrs = at; cfg.numAttrs = n;
    return cudaLaunchKernelEx(&cfg, kernel, std::forward<Args>(args)...);
}
template <typename... KArgs, typename... Args>
cudaError_t launch_k(void (*kernel)(KArgs...), unsigned grid, unsigned block, size_t smem, cudaStream_t s, int pdl_max,
                     Args&&... args) {
    return launch_k(kernel, dim3(grid), block, smem, s, pdl_max, std::forward<Args>(args)...);
}

// Partial right-looking Cholesky of the leading T_elim block columns of a T_total-block lower matrix
// (T_elim == T_total: plain Cholesky).  The trailing block is left holding the Schur complement.
//
// Panels are processed in GROUPS of G (2 or 4): inside a group, before panel g is factored its block column gets
// ONE update with all the group's earlier panels (left-looking, K = 128 g, 2R tiles); after the last panel the
// trailing matrix gets ONE rank-128G update with [P_0 | ... | P_{G-1}], which divides the read-modify-write
// traffic and the per-tile overhead of the dominant kernel by G.
// Look-ahead: the big update first covers the next group's block columns (part 1); the next group's head
// (potrf, trsm, column update, ...) then runs on the side stream under the rest of the update.
//
// identity_border: the border is the identity in data order (m = n, border row a is 1 at column pad + a; the gradient
// entries).  C L^-T is then upper triangular, so border row block T_elim + b is zero in every panel before panel b, and
// in the panel group that ends at block g1 only border row blocks [T_elim, T_elim + g1) are non-zero.  Every launch of
// group q (the panel solves, the in-group column updates, both parts of the group update and the residual blocks) then
// ends at row block T_elim + gstart[q + 1] instead of T_total: the rows it leaves out would only subtract exact zeros.
// Each panel solve of a group covers up to the group's end, not only its own reach, because the group update reads the
// group's panels side by side.  The elimination drops from 7 N^3 / 3 to N^3 flops.  Tile shapes, the group size, the
// chain and the yield mode are still chosen from T_total, and every tile runs the same k loop as without the
// restriction: the trailing block and the residual are the same bits.
//
// envelope (T_elim == T_total only; may be null): envelope[e] (fill.cuh envelope_kernel, on the device) is the first row
// block from which every row is exactly zero in block columns [0, e) of the filled matrix.  Cholesky keeps a row's
// leading zeros (L_ij = 0 for j before the row's first non-zero in K), so in the group that ends at panel e those rows
// have exact-zero panel-solve inputs, exact +0 panels, and every product they would take part in has a +-0 factor:
// the update C - 0 leaves C as it is, except that the sign of a zero can differ inside entries that stay zero and are
// never pivoted.  The kernels read the entry after pdl_wait() and stop their rows there (gemm.cuh row_limit); the grids,
// the group boundaries and every other host-side choice stay those of the full launch, which bound them from above.
// The likelihood is the same bits as the unrestricted factorisation in the same row order.  Rows sorted by wavelength
// give a narrow envelope (squared-exponential entries underflow to +0 beyond about 38.6 length scales); in any other
// order it is T_total everywhere and every launch runs in full.
int launch_factor(const Lanes& ln, double* W, int64_t ld, int T_elim, int T_total, int pad, const FactorWs& ws,
                  const int* sentinel, double* result, bool identity_border = false, const int* envelope = nullptr) {
    const int64_t ldp = ws.Nt;
    CUtensorMap mapW, mapLinv, mapPa[2], mapPb[2], mapPas[2], mapPbs[2];   // ..s: boxes of the small tile shape
    CUtensorMap mapWblk, mapWt, mapL7[3];                                   // chain 7: diagonal block, panel tile, L_kk below its sub-blocks
    {
        const uint64_t Nt = (uint64_t)T_total * NB;
        int rcm = make_tensor_map(&mapW, W, Nt, Nt, (uint64_t)ld, SA);
        if (!rcm) rcm = make_tensor_map(&mapLinv, ws.Linv, NB, NB, NB, SB);
        if (!rcm) rcm = make_tensor_map(&mapWblk, W, Nt, Nt, (uint64_t)ld, P7_LD, NB);
        if (!rcm) rcm = make_tensor_map(&mapWt, W, Nt, Nt, (uint64_t)ld, T7_RS, NB);
        if (!rcm) rcm = make_tensor_map(&mapL7[0], ws.Linv, NB, NB, NB, T7_LS0, 32);
        if (!rcm) rcm = make_tensor_map(&mapL7[1], ws.Linv, NB, NB, NB, T7_LS1, 32);
        if (!rcm) rcm = make_tensor_map(&mapL7[2], ws.Linv, NB, NB, NB, T7_LS2, 32);
        for (int q = 0; q < 2 && !rcm; ++q) {
            rcm = make_tensor_map(&mapPa[q], ws.P[q], (uint64_t)ldp, (uint64_t)MAX_GROUP * NB, (uint64_t)ldp, SA);
            if (!rcm) rcm = make_tensor_map(&mapPb[q], ws.P[q], (uint64_t)ldp, (uint64_t)MAX_GROUP * NB, (uint64_t)ldp, SB);
            if (!rcm) rcm = make_tensor_map(&mapPas[q], ws.P[q], (uint64_t)ldp, (uint64_t)MAX_GROUP * NB, (uint64_t)ldp, Shape<2>::SA);
            if (!rcm) rcm = make_tensor_map(&mapPbs[q], ws.P[q], (uint64_t)ldp, (uint64_t)MAX_GROUP * NB, (uint64_t)ldp, Shape<2>::SB);
        }
        if (rcm) return rcm;
    }
    // Wide updates are worth their longer panel chain when that chain is hidden anyway: the graph farm runs rank-1024
    // updates (G = 8: C4 4.62 -> 4.66 evals/s against G = 4 with 64 branches; G = 4 against 2 was 4.30 -> 4.37 in round 1), a
    // large matrix rank-512 (N = 16384: 50.0 -> 49.1 ms); a single mid-size matrix is faster with G = 2 (N = 9000: 11.2 vs
    // 11.7 ms).
    const int G = g_group ? g_group : (ln.group ? ln.group : (T_total >= 96 ? 4 : 2));
    auto pbuf = [&](int q) { return ws.P[q & 1]; };
    auto kbeg_of = [&](int q) { return q == 0 ? (pad / BK) * BK : 0; };
    // a very large matrix has hundreds of 32-row panel-solve tiles per panel: the GEMM panel solve wins again
    // (N = 32768: 342 vs 350 ms)
    const int chain = ln.chain ? ln.chain : (T_total >= 192 ? 3 : g_potrf_version);
    auto potrf = [&](cudaStream_t s, int kb) {
        if (chain == 7)   // blocked: one chain warp, DMMA followers and rank-32 updates (chain.cuh, experimental)
            launch_k(potrf_diag7_kernel, 1, P7_THREADS, POTRF7_SMEM, s, ln.pdl, (const double*)W, ld, kb, pad, ws.Linv,
                     ws.Xd, ws.rvec, ws.y + (int64_t)kb * NB, ws.acc, ws.info, sentinel, (int)(kb == T_elim - 1), result, mapWblk);
        else
            launch_k(potrf_diag3_kernel, 1, 256, POTRF_SMEM, s, ln.pdl, (const double*)W, ld, kb, pad, ws.Linv, ws.rvec,
                     ws.y + (int64_t)kb * NB, ws.acc, ws.info, sentinel, (int)(kb == T_elim - 1), result);
    };
    // last row block (exclusive) of the launches of group q; set once the group boundaries are known
    std::vector<int> tend;
    std::vector<int> gstart;
    auto trsm = [&](cudaStream_t s, int kb, int q, int col0) {
        const int R = tend[q] - kb - 1;
        if (chain == 7) {   // blocked substitution against L_kk and its 32 x 32 diagonal inverses (chain.cuh)
            Trsm7Args a;
            a.W = W; a.ld = ld; a.kb = kb; a.Lfac = ws.Linv; a.Xd = ws.Xd;
            a.P = pbuf(q) + (int64_t)col0 * ldp; a.ldp = ldp; a.ntiles = 4 * R;
            a.tend = envelope; a.tend_at = gstart[q + 1];
            launch_k(trsm7_kernel, std::min(4 * R, g_num_sms), T7_THREADS, TRSM7_SMEM, s, ln.pdl, a, mapWt, mapL7[0], mapL7[1],
                     mapL7[2]);
            return;
        }
        TrsmSrc src;
        src.W = W; src.ld = ld; src.kb = kb; src.kbeg = (kb == 0) ? (pad / BK) * BK : 0;
        src.Linv = ws.Linv; src.P = pbuf(q) + (int64_t)col0 * ldp; src.ldp = ldp;
        src.tend = envelope; src.tend_at = gstart[q + 1];
        launch_k(trsm3_kernel, persistent_ctas(2 * R), 256, GEMM_SMEM, s, ln.pdl, src, 2 * R, mapW, mapLinv);
    };
    // update of row tiles [row0, T_total) with k range [kbeg, kend) of group buffer q; the residual blocks (if
    // ykb >= 0) apply panel ykb, whose columns start at res_col0 in the buffer
    auto syrk = [&](cudaStream_t s, int q, int row0, int kend, int part, int ncol1, int ykb, int res_col0) {
        const int R = tend[q] - row0;
        // part 1 (the block columns the next diagonal blocks wait for) of a matrix factored on its own: 64 x 32 tiles,
        // four times the CTAs at a quarter of the latency each
        const int sh = (part == 1 && chain == 7) ? 2 : 1;
        SyrkSrc src;
        src.W = W; src.ld = ld; src.row0 = sh * row0; src.res_row0 = row0; src.kbeg = kbeg_of(q); src.kend = kend;
        src.P = pbuf(q); src.ldp = ldp; src.part = part; src.ncol1 = sh * ncol1;
        src.tend = envelope; src.tend_at = gstart[q + 1];
        const int ntiles = syrk_ntiles(sh * R, part, sh * ncol1);
        const int nres = (part == 2 || ykb < 0) ? 0 : R;
        if (ntiles + nres == 0) return;
        // Under look-ahead the bulk update (part 2) must leave room for the links of the next group (high-priority side
        // stream).  Mode 2: it stays persistent but takes ONE slot per SM and leaves one SM empty, so that every link
        // finds a slot on every SM at once (a panel-solve CTA, 126 KB of shared memory, fits beside an update CTA,
        // 102 KB, and not beside two) and the one-CTA diagonal block, which needs a whole SM's shared memory, an empty SM
        // instead of waiting 20-40 us for two update CTAs to retire.  Mode 1: one tile per CTA on all slots, which free
        // up continuously.  N = 4000 / 6000 / 9000: 1.70 / 3.50 / 9.31 ms in mode 2, 1.75 / 3.64 / 9.39 in mode 1; where
        // the bulk dominates mode 1 wins (N = 16384: 47.4 vs 47.7 ms, N = 32768: 349 vs 364 ms), so by default mode 2
        // below 96 panels and mode 1 from there.
        const int yield_mode = g_yield_lookahead ? g_yield_lookahead : (T_total >= 96 ? 1 : 2);
        const bool yield_slots = (part == 2 && ln.side != nullptr);
        const double* yk = ws.y + (int64_t)std::max(ykb, 0) * NB;
        if (sh == 2) {
            const int nctas = persistent_ctas(ntiles);
            launch_k(syrk3_kernel<2>, nctas + nres, 256, Shape<2>::SMEM, s, ln.pdl, src, ntiles, nctas, nres, yk, ws.rvec,
                     res_col0, mapPas[q & 1], mapPbs[q & 1], mapPas[q & 1], mapPbs[q & 1]);
        } else {
            SyrkSplit sp = syrk_split(ntiles, yield_slots && yield_mode == 1, part != 1 && g_tail_split != 0);
            if (yield_slots && yield_mode == 2) sp.nctas = std::min(sp.nmain, g_num_sms - 1);
            launch_k(syrk3_kernel<1>, nres + sp.nctas + sp.nquarters, 256, sp.nquarters ? SYRK1_SMEM : GEMM_SMEM, s, ln.pdl, src, sp.nmain, sp.nctas, nres,
                     yk, ws.rvec, res_col0, mapPa[q & 1], mapPb[q & 1], mapPas[q & 1], mapPbs[q & 1]);
        }
        ++g_launches;
    };
    // Group boundaries.  Uniform groups of G, except at the END of a matrix factored on its own (look-ahead, chain 7):
    // once fewer than SINGLE_ROWS row blocks remain the trailing update is shorter than the links it runs beside,
    // the chain is all there is, and single panels (no in-group column update, a rank-128 update of ONE block column
    // before the next diagonal block) make the shortest chain: 38 us per panel against 48.  Measured with 0 / 16 / 24 / 36
    // such rows: N = 4000 1.706 / 1.675 / 1.647 / 1.625 ms, N = 6000 3.514 / 3.491 / 3.442 / 3.526, N = 9000 9.31 / 9.29 / 9.25 / 9.33.
    constexpr int SINGLE_ROWS = 24;
    {
        const bool lone = ln.side != nullptr && chain == 7 && g_group == 0;
        for (int a = 0; a < T_elim;) {
            const int g = (lone && T_total - a <= SINGLE_ROWS) ? 1 : G;
            gstart.push_back(a);
            a += std::min(g, T_elim - a);
        }
        gstart.push_back(T_elim);
    }
    const int ngroups = (int)gstart.size() - 1;
    for (int q = 0; q < ngroups; ++q) tend.push_back(identity_border ? T_elim + gstart[q + 1] : T_total);
    auto group_size = [&](int q) { return gstart[q + 1] - gstart[q]; };
    // everything of group q that precedes its big update: for each panel g: (column update with the group's
    // earlier panels, which also carries the residual update of panel g-1), potrf, trsm
    auto head = [&](cudaStream_t s, int q) -> int {
        const int a = gstart[q], n = group_size(q);
        for (int g = 0; g < n; ++g) {
            const int kb = a + g;
            if (g > 0) syrk(s, q, kb, g * NB, 1, 2, kb - 1, (g - 1) * NB);   // block column kb, K = 128 g
            potrf(s, kb); LAUNCH_CHECK();
            if (tend[q] - kb - 1 > 0) { trsm(s, kb, q, g * NB); LAUNCH_CHECK(); }
        }
        return PSOAP_OK;
    };
    // the big update of group q with all its panels (the residual blocks apply its last panel)
    auto update = [&](cudaStream_t s, int q, int part, int ncol1) {
        const int a = gstart[q], n = group_size(q);
        syrk(s, q, a + n, n * NB, part, ncol1, a + n - 1, (n - 1) * NB);
    };
    int rc = head(ln.main, 0);
    if (rc) return rc;
    for (int q = 0; q < ngroups; ++q) {
        const bool next = q + 1 < ngroups;
        if (!next || ln.side == nullptr) {
            update(ln.main, q, 0, 2);
            if (next) { rc = head(ln.main, q + 1); if (rc) return rc; }
            continue;
        }
        const int ncol1 = 2 * group_size(q + 1);   // block columns the next group's head touches
        update(ln.main, q, 1, ncol1);
        CUDA_TRY(cudaEventRecord(ln.e1, ln.main));
        CUDA_TRY(cudaStreamWaitEvent(ln.side, ln.e1, 0));
        rc = head(ln.side, q + 1);
        if (rc) return rc;
        CUDA_TRY(cudaEventRecord(ln.e2, ln.side));
        update(ln.main, q, 2, ncol1);
        CUDA_TRY(cudaStreamWaitEvent(ln.main, ln.e2, 0));
    }
    cudaError_t e_ = cudaGetLastError();
    if (e_ != cudaSuccess) return fail(PSOAP_ERR_CUDA, std::string("launch: ") + cudaGetErrorString(e_));
    return PSOAP_OK;
}

// Calls fn(nc) with nc a std::integral_constant<int, ncomp> (1, 2 or 3): the one place where a run-time number of
// components picks the instantiation of a kernel template.
template <class Fn>
void with_ncomp(int ncomp, Fn&& fn) {
    if (ncomp == 1) fn(std::integral_constant<int, 1>{});
    else if (ncomp == 2) fn(std::integral_constant<int, 2>{});
    else fn(std::integral_constant<int, 3>{});
}

int launch_fill_lower(int ncomp, cudaStream_t st, double* W, int64_t ld, int T, int pad, const ZSource& zs,
                      const double* sigma, const double* fl, double mu, const GpParams& gp, const FactorWs& ws) {
    with_ncomp(ncomp, [&](auto nc) {
        launch_k(fill_lower_kernel<nc>, (unsigned)(T * (T + 1) / 2), 256, 0, st, 0, W, ld, pad, zs, sigma, fl, mu, gp,
                 ws.rvec, ws.acc, ws.info, ws.nz);
    });
    LAUNCH_CHECK();
    return PSOAP_OK;
}

// fill + factor + fused solve of one chunk on stream st
int launch_chunk(const Lanes& ln, int ncomp, int64_t N, const ZSource& zs, const double* fl, const double* sigma,
                 double mu, const GpParams& gp, const FactorWs& ws, const int* sentinel, double* result) {
    const int64_t Np = padded_dim(N);
    const int T = (int)(Np / NB);
    const int pad = (int)(Np - N);
    int rc = launch_fill_lower(ncomp, ln.main, ws.W, Np, T, pad, zs, sigma, fl, mu, gp, ws);
    if (rc) return rc;
    if (T > ENV_MAX_T) return fail(PSOAP_ERR_ARG, "launch_chunk: matrix too large for the envelope");
    launch_k(envelope_kernel, 1, 256, 0, ln.main, ln.pdl, (const uint8_t*)ws.nz, T, ws.tend);
    LAUNCH_CHECK();
    return launch_factor(ln, ws.W, Np, T, T, pad, ws, sentinel, result, false, ws.tend);
}

// Side stream + events for calls on a caller-provided stream (one set per host thread).
struct SideLane {
    cudaStream_t side = nullptr;
    cudaEvent_t e1 = nullptr, e2 = nullptr;
};
int get_lanes(cudaStream_t user, Lanes* ln) {
    thread_local SideLane sl;
    if (!sl.side) {
        int lo = 0, hi = 0;
        CUDA_TRY(cudaDeviceGetStreamPriorityRange(&lo, &hi));
        CUDA_TRY(cudaStreamCreateWithPriority(&sl.side, cudaStreamNonBlocking, hi));
        CUDA_TRY(cudaEventCreateWithFlags(&sl.e1, cudaEventDisableTiming));
        CUDA_TRY(cudaEventCreateWithFlags(&sl.e2, cudaEventDisableTiming));
    }
    // g_lookahead / g_pdl were read from the environment once, in set_kernel_attributes()
    ln->main = user; ln->side = g_lookahead ? sl.side : nullptr; ln->e1 = sl.e1; ln->e2 = sl.e2;
    ln->pdl = g_pdl;
    return PSOAP_OK;
}

__global__ void write_result_kernel(double* result, double lnlike, double logdet, double quad, double info) {
    result[0] = lnlike; result[1] = logdet; result[2] = quad; result[3] = info;
}

// GP hyper-parameters read on the device from dev ([amp, l] per component; null: from amp / l), unused components inert
GpParams gp_params(const double* dev) {
    GpParams gp;
    gp.dev = dev;
    for (int c = 0; c < 3; ++c) { gp.amp[c] = 0; gp.l[c] = 1; }
    return gp;
}

bool make_gp(int ncomp, const double* amp, const double* l, GpParams* gp) {
    bool neg = false;
    *gp = gp_params(nullptr);
    for (int c = 0; c < ncomp; ++c) {
        gp->amp[c] = amp[c];
        gp->l[c] = l[c];
        if (amp[c] < 0.0 || l[c] < 0.0) neg = true;
    }
    return neg;
}

ZSource direct_z(const double* f, const double* g, const double* h) {
    ZSource zs;
    zs.lwl[0] = f; zs.lwl[1] = g; zs.lwl[2] = h;
    zs.epoch = nullptr; zs.vel = nullptr; zs.n_epochs = 0; zs.shift = 0;
    return zs;
}

// the chunk's pixels shifted by a velocity table on the device [ncomp][n_epochs], as the farm and the chunk entries read them
ZSource farm_z(const psoap_chunk& ch, const double* vel) {
    ZSource zs = direct_z(ch.lwl, nullptr, nullptr);
    zs.epoch = ch.epoch; zs.vel = vel; zs.n_epochs = ch.n_epochs; zs.shift = 1;
    return zs;
}

}  // namespace

// ======================================================================================================
extern "C" {

const char* psoap_last_error(void) { return g_err.c_str(); }
int psoap_version(void) { return 104; }
int psoap_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}
int64_t psoap_launch_count(void) { return g_launches.load(); }
int psoap_model_ncomp(int model) { return (model >= 1 && model <= 5) ? model_ncomp(model) : 0; }
int psoap_model_norb(int model) { return (model >= 1 && model <= 5) ? model_norb(model) : 0; }

// ---- fills ------------------------------------------------------------------------------------------
int psoap_fill_v11(int ncomp, double* mat, int64_t ld, int64_t N, const double* lwl_f, const double* lwl_g,
                   const double* lwl_h, const double* amp, const double* l, void* stream) {
    if (ncomp < 1 || ncomp > 3 || !mat || !lwl_f || (ncomp > 1 && !lwl_g) || (ncomp > 2 && !lwl_h) || ld < N || N < 0 ||
        N > (1 << 30))
        return fail(PSOAP_ERR_ARG, "psoap_fill_v11: bad arguments");
    if (N == 0) return PSOAP_OK;
    GpParams gp;
    make_gp(ncomp, amp, l, &gp);
    ZSource zs = direct_z(lwl_f, lwl_g, lwl_h);
    cudaStream_t st = (cudaStream_t)stream;
    const int T = (int)((N + 63) / 64);
    const unsigned grid = (unsigned)((int64_t)T * (T + 1) / 2);
    with_ncomp(ncomp, [&](auto nc) { fill_full_kernel<nc><<<grid, 256, 0, st>>>(mat, ld, (int)N, zs, gp); });
    LAUNCH_CHECK();
    return PSOAP_OK;
}

// fill_V11_* for HOST arrays (synchronous): what a Cython/ctypes seam at matrix_functions.pyx binds when the caller's
// `mat` and ln-wavelength vectors live in host memory.  The N x N result crosses PCIe; the likelihood never needs this.
int psoap_fill_v11_host(int ncomp, double* mat, int64_t ld, int64_t N, const double* lwl_f, const double* lwl_g,
                        const double* lwl_h, const double* amp, const double* l) {
    if (ncomp < 1 || ncomp > 3 || !mat || !lwl_f || (ncomp > 1 && !lwl_g) || (ncomp > 2 && !lwl_h) || ld < N || N < 0 ||
        N > (1 << 30) || !amp || !l)
        return fail(PSOAP_ERR_ARG, "psoap_fill_v11_host: bad arguments");
    if (N == 0) return PSOAP_OK;
    const size_t vec = align_up((size_t)N * 8, 256);
    char* base = nullptr;
    CUDA_TRY(cudaMalloc(&base, (size_t)N * N * 8 + 3 * vec));
    double* dmat = (double*)base;
    double* dv[3];
    const double* hv[3] = {lwl_f, lwl_g, lwl_h};
    cudaError_t e = cudaSuccess;
    for (int c = 0; c < 3; ++c) {
        dv[c] = (double*)(base + (size_t)N * N * 8 + c * vec);
        if (c < ncomp && e == cudaSuccess) e = cudaMemcpy(dv[c], hv[c], (size_t)N * 8, cudaMemcpyHostToDevice);
    }
    int rc = PSOAP_OK;
    if (e == cudaSuccess)
        rc = psoap_fill_v11(ncomp, dmat, N, N, dv[0], ncomp > 1 ? dv[1] : nullptr, ncomp > 2 ? dv[2] : nullptr, amp, l, nullptr);
    if (e == cudaSuccess && rc == PSOAP_OK)
        e = cudaMemcpy2D(mat, (size_t)ld * 8, dmat, (size_t)N * 8, (size_t)N * 8, (size_t)N, cudaMemcpyDeviceToHost);
    cudaFree(base);
    if (rc) return rc;
    if (e != cudaSuccess) return fail(PSOAP_ERR_CUDA, std::string("psoap_fill_v11_host: ") + cudaGetErrorString(e));
    return PSOAP_OK;
}

int psoap_fill_v12n(int ncomp, double* mat, int64_t ld, int64_t M, int64_t N, const double* const* rows,
                    const double* const* cols, const double* amp, const double* l, void* stream) {
    if (ncomp < 1 || ncomp > 3 || !mat || !rows || !cols || !amp || !l || ld < N || M < 0 || N < 0)
        return fail(PSOAP_ERR_ARG, "psoap_fill_v12n: bad arguments");
    if (M == 0 || N == 0) return PSOAP_OK;
    GpParams gp;
    make_gp(ncomp, amp, l, &gp);
    V12Src src;
    for (int c = 0; c < 3; ++c) {
        src.rows[c] = c < ncomp ? rows[c] : nullptr;
        src.cols[c] = c < ncomp ? cols[c] : nullptr;
        if (c < ncomp && (!rows[c] || !cols[c])) return fail(PSOAP_ERR_ARG, "psoap_fill_v12n: null vector");
    }
    dim3 grid((unsigned)((N + 63) / 64), (unsigned)((M + 63) / 64));
    cudaStream_t st = (cudaStream_t)stream;
    with_ncomp(ncomp, [&](auto nc) { fill_v12_kernel<nc><<<grid, 256, 0, st>>>(mat, ld, (int)M, (int)N, src, gp); });
    LAUNCH_CHECK();
    return PSOAP_OK;
}

int psoap_fill_v12(double* mat, int64_t ld, int64_t M, int64_t N, const double* rows, const double* cols, double amp,
                   double l, void* stream) {
    return psoap_fill_v12n(1, mat, ld, M, N, &rows, &cols, &amp, &l, stream);
}

int psoap_replicate_wls(double* out, const double* lwl, const int32_t* epoch, int64_t N, const double* vel, int ncomp,
                        int n_epochs, void* stream) {
    if (!out || !lwl || !epoch || !vel || ncomp < 1 || ncomp > 3 || N < 0)
        return fail(PSOAP_ERR_ARG, "psoap_replicate_wls: bad arguments");
    if (N == 0) return PSOAP_OK;
    ZSource zs = direct_z(lwl, nullptr, nullptr);
    zs.epoch = epoch; zs.vel = vel; zs.n_epochs = n_epochs; zs.shift = 1;
    replicate_wls_kernel<<<(unsigned)((N + 255) / 256), 256, 0, (cudaStream_t)stream>>>(out, zs, N, ncomp);
    LAUNCH_CHECK();
    return PSOAP_OK;
}

int psoap_orbit_velocities(int model, const double* p_orb, const double* dates, int n_epochs, double* vel, int* flag,
                           void* stream) {
    if (model < 1 || model > 5 || !p_orb || !dates || !vel || n_epochs < 0)
        return fail(PSOAP_ERR_ARG, "psoap_orbit_velocities: bad arguments");
    if (n_epochs == 0) return PSOAP_OK;
    orbit_kernel<<<1, 128, 0, (cudaStream_t)stream>>>(model, p_orb, dates, n_epochs, vel, flag, 0);
    LAUNCH_CHECK();
    return PSOAP_OK;
}

// ---- likelihood -------------------------------------------------------------------------------------
size_t psoap_lnlike_workspace_bytes(int64_t N) { return factor_ws_bytes(padded_dim(std::max<int64_t>(N, 1))); }

int psoap_lnlike(int ncomp, int64_t N, const double* lwl_f, const double* lwl_g, const double* lwl_h, const double* fl,
                 const double* sigma, const double* amp, const double* l, double mu_GP, void* workspace,
                 size_t workspace_bytes, psoap_result* result, void* stream) {
    if (ncomp < 1 || ncomp > 3 || N < 0 || N > 200000 || !amp || !l || !result)
        return fail(PSOAP_ERR_ARG, "psoap_lnlike: bad arguments");
    cudaStream_t st = (cudaStream_t)stream;
    GpParams gp;
    if (make_gp(ncomp, amp, l, &gp)) {  // covariance.py:317-318: negative hyper-parameters -> -inf
        write_result_kernel<<<1, 1, 0, st>>>((double*)result, -INFINITY, 0.0, 0.0, 0.0);
        LAUNCH_CHECK();
        return PSOAP_OK;
    }
    if (N == 0) {  // empty chunk: the reference's sums run over nothing, -0.5 * (0 + 0) = -0.0
        write_result_kernel<<<1, 1, 0, st>>>((double*)result, -0.0, 0.0, 0.0, 0.0);
        LAUNCH_CHECK();
        return PSOAP_OK;
    }
    if (!lwl_f || (ncomp > 1 && !lwl_g) || (ncomp > 2 && !lwl_h) || !fl || !sigma)
        return fail(PSOAP_ERR_ARG, "psoap_lnlike: null vector");
    if (!workspace || workspace_bytes < psoap_lnlike_workspace_bytes(N) || ((uintptr_t)workspace & 255))
        return fail(PSOAP_ERR_WORKSPACE, "psoap_lnlike: workspace too small or not 256-byte aligned");
    int rc = set_kernel_attributes();
    if (rc) return rc;
    FactorWs ws;
    carve_factor_ws((char*)workspace, padded_dim(N), &ws, true);
    Lanes ln;
    rc = get_lanes(st, &ln);
    if (rc) return rc;
    return launch_chunk(ln, ncomp, N, direct_z(lwl_f, lwl_g, lwl_h), fl, sigma, mu_GP, gp, ws, nullptr, (double*)result);
}

int psoap_lnlike_envelope_view(void* workspace, int64_t N, int** tend, int* T) {
    if (!workspace || N < 1 || !tend || !T) return fail(PSOAP_ERR_ARG, "psoap_lnlike_envelope_view: bad arguments");
    FactorWs ws;
    carve_factor_ws((char*)workspace, padded_dim(N), &ws, true);
    *tend = ws.tend;
    *T = (int)(padded_dim(N) / NB);
    return PSOAP_OK;
}

namespace {
struct HostCache {
    std::mutex mu;
    void* buf = nullptr;
    size_t bytes = 0;
    cudaStream_t st = nullptr;
} g_hc;
}

int psoap_lnlike_host(int ncomp, int64_t N, const double* lwl_f, const double* lwl_g, const double* lwl_h,
                      const double* fl, const double* sigma, const double* amp, const double* l, double mu_GP,
                      psoap_result* result) {
    if (ncomp < 1 || ncomp > 3 || N < 0 || !amp || !l || !result)
        return fail(PSOAP_ERR_ARG, "psoap_lnlike_host: bad arguments");
    if (N == 0) {  // empty chunk (see psoap_lnlike); no device work
        GpParams gp;
        result->lnlike = make_gp(ncomp, amp, l, &gp) ? -INFINITY : -0.0;
        result->logdet = result->quad = result->info = 0.0;
        return PSOAP_OK;
    }
    if (!lwl_f || !fl || !sigma || (ncomp > 1 && !lwl_g) || (ncomp > 2 && !lwl_h))
        return fail(PSOAP_ERR_ARG, "psoap_lnlike_host: null vector");
    std::lock_guard<std::mutex> lock(g_hc.mu);
    const size_t vec = align_up((size_t)N * 8, 256);
    const size_t need = psoap_lnlike_workspace_bytes(N) + 5 * vec + 256;
    if (g_hc.bytes < need) {
        if (g_hc.buf) cudaFree(g_hc.buf);
        g_hc.buf = nullptr; g_hc.bytes = 0;
        CUDA_TRY(cudaMalloc(&g_hc.buf, need));
        g_hc.bytes = need;
    }
    if (!g_hc.st) CUDA_TRY(cudaStreamCreateWithFlags(&g_hc.st, cudaStreamNonBlocking));
    char* base = (char*)g_hc.buf;
    double* d[5];
    const double* h[5] = {lwl_f, lwl_g, lwl_h, fl, sigma};
    for (int i = 0; i < 5; ++i) {
        d[i] = (double*)(base + i * vec);
        if (h[i] && (i >= 3 || i < ncomp)) CUDA_TRY(cudaMemcpyAsync(d[i], h[i], (size_t)N * 8, cudaMemcpyHostToDevice, g_hc.st));
    }
    psoap_result* dres = (psoap_result*)(base + 5 * vec);
    void* wsp = base + 5 * vec + 256;
    int rc = psoap_lnlike(ncomp, N, d[0], ncomp > 1 ? d[1] : nullptr, ncomp > 2 ? d[2] : nullptr, d[3], d[4], amp, l, mu_GP,
                          wsp, g_hc.bytes - 5 * vec - 256, dres, g_hc.st);
    if (rc) return rc;
    CUDA_TRY(cudaMemcpyAsync(result, dres, sizeof(psoap_result), cudaMemcpyDeviceToHost, g_hc.st));
    CUDA_TRY(cudaStreamSynchronize(g_hc.st));
    return PSOAP_OK;
}

// ---- Schur complement of a bordered matrix (prediction) -----------------------------------------------
size_t psoap_schur_workspace_bytes(int64_t n, int64_t m) {
    const int64_t Nt = padded_dim(n) + padded_dim(std::max<int64_t>(m, 0));
    return factor_ws_bytes(Nt) - align_up((size_t)Nt * Nt * 8, 256);
}

// S: column-major [Nt, ld] with Nt = padded(n) + padded(m).  The caller lays the leading block out with
// FRONT padding (identity in the first padded(n) - n rows/cols) and the border from row padded(n) on;
// rows beyond padded(n) + m are dead padding.  rvec (residual over all Nt rows) is taken from / returned in
// the workspace through psoap_schur_residual.
int psoap_schur(double* S, int64_t ld, int64_t n, int64_t m, void* workspace, size_t workspace_bytes,
                psoap_result* result, void* stream) {
    if (!S || n < 1 || m < 0 || !workspace || !result) return fail(PSOAP_ERR_ARG, "psoap_schur: bad arguments");
    const int64_t Nn = padded_dim(n), Nt = Nn + padded_dim(m);
    if (ld < Nt || (ld & 1) || ((uintptr_t)S & 15)) return fail(PSOAP_ERR_ARG, "psoap_schur: ld/alignment");
    if (workspace_bytes < psoap_schur_workspace_bytes(n, m) || ((uintptr_t)workspace & 255))
        return fail(PSOAP_ERR_WORKSPACE, "psoap_schur: workspace too small or misaligned");
    int rc = set_kernel_attributes();
    if (rc) return rc;
    FactorWs ws;
    carve_factor_ws((char*)workspace, Nt, &ws, false);
    Lanes ln;
    rc = get_lanes((cudaStream_t)stream, &ln);
    if (rc) return rc;
    return launch_factor(ln, S, ld, (int)(Nn / NB), (int)(Nt / NB), (int)(Nn - n), ws, nullptr, (double*)result);
}

}  // extern "C"

// The residual / accumulator part of a Schur workspace, for the host-side prediction code.
extern "C" int psoap_schur_views(void* workspace, int64_t n, int64_t m, double** rvec, double** acc, int** info) {
    const int64_t Nt = padded_dim(n) + padded_dim(std::max<int64_t>(m, 0));
    FactorWs ws;
    carve_factor_ws((char*)workspace, Nt, &ws, false);
    if (rvec) *rvec = ws.rvec;
    if (acc) *acc = ws.acc;
    if (info) *info = ws.info;
    return PSOAP_OK;
}

// ---- gradient of the log-likelihood (grad.cuh) -----------------------------------------------------------
namespace {
// The gradient entries factor the identity-bordered matrix S = [[K, I], [I, 0]]: data block front-padded to Nn, a
// border of Nn rows after it (no front padding), Nt = 2 Nn.  Workspace: S and the factorisation scratch first, so
// that their offsets depend on N alone (psoap_lnlike_grad_views), then the contraction partials, then (chunk entry)
// the velocity table, sentinel, orbit Jacobian and the per-pixel / per-epoch gradients.
struct GradWs {
    double* S;
    FactorWs f;
    double* tile;   // [ntiles][2 ncomp]
    double* slot;   // [Tb][Tb][ncomp][128]
    double* hyp;    // [2 ncomp + 1]
    double* vel;    // [3][n_epochs]
    int* flag;
    double* jac;    // [3][n_epochs][norb]
    double* gz;     // [ncomp][N]
    double* gv;     // [3][n_epochs]
    int64_t Nn, Nt;
    int Tb, ntiles;
};
size_t carve_grad_ws(char* base, int ncomp, int64_t N, int n_epochs, int norb, GradWs* g) {
    g->Nn = padded_dim(std::max<int64_t>(N, 1));
    g->Nt = 2 * g->Nn;
    g->Tb = (int)(g->Nn / NB);
    g->ntiles = g->Tb * (g->Tb + 1) / 2;
    size_t off = 0;
    auto take = [&](size_t bytes) { char* r = base ? base + off : nullptr; off += align_up(bytes, 256); return r; };
    g->S = (double*)take((size_t)g->Nt * g->Nt * 8);
    const size_t fbytes = factor_ws_bytes(g->Nt) - align_up((size_t)g->Nt * g->Nt * 8, 256);
    char* fb = take(fbytes);
    if (base) carve_factor_ws(fb, g->Nt, &g->f, false);
    g->tile = (double*)take((size_t)g->ntiles * 2 * ncomp * 8);
    g->slot = (double*)take((size_t)g->Tb * g->Tb * ncomp * NB * 8);
    g->hyp = (double*)take(8 * 8);
    g->vel = (double*)take((size_t)3 * n_epochs * 8);
    g->flag = (int*)take(4);
    g->jac = (double*)take((size_t)3 * n_epochs * norb * 8);
    g->gz = (double*)take((size_t)ncomp * N * 8);
    g->gv = (double*)take((size_t)3 * n_epochs * 8);
    return off;
}

// fill, identity border, restricted elimination, contraction and the hyper-parameter reduction (+ the per-pixel
// gradient when grad_z is given) of one problem on ln.main
int launch_grad(const Lanes& ln, int ncomp, int64_t N, const ZSource& zs, const double* fl, const double* sigma,
                double mu, const GpParams& gp, const GradWs& g, const int* sentinel, double* result, double* grad_hyp,
                double* grad_z) {
    const int Tn = (int)(g.Nn / NB), Tt = 2 * Tn, pad = (int)(g.Nn - N);
    cudaStream_t st = ln.main;
    int rc = launch_fill_lower(ncomp, st, g.S, g.Nt, Tn, pad, zs, sigma, fl, mu, gp, g.f);
    if (rc) return rc;
    const unsigned nborder = (unsigned)((int64_t)Tt * (Tt + 1) / 2 - (int64_t)Tn * (Tn + 1) / 2);
    grad_border_kernel<<<nborder, 256, 0, st>>>(g.S, g.Nt, (int)g.Nn, (int)N, pad, g.f.rvec);
    LAUNCH_CHECK();
    rc = launch_factor(ln, g.S, g.Nt, Tn, Tt, pad, g.f, sentinel, result, true);
    if (rc) return rc;
    const GradOut out{g.tile, g.slot, g.Tb};
    with_ncomp(ncomp, [&](auto nc) {
        lnlike_grad_kernel<nc><<<g.ntiles, 256, 0, st>>>(g.S, g.Nt, (int)g.Nn, (int)N, g.f.rvec, zs, gp, out);
    });
    LAUNCH_CHECK();
    grad_hyp_kernel<<<1, 256, 0, st>>>(g.tile, g.ntiles, ncomp, g.f.rvec, (int)g.Nn, (int)N, gp, g.f.info, sentinel, grad_hyp);
    LAUNCH_CHECK();
    if (grad_z) {
        grad_pixel_kernel<<<(unsigned)(ncomp * g.Tb), NB, 0, st>>>(g.slot, g.Tb, ncomp, (int)N, gp, g.f.info, sentinel, grad_z);
        LAUNCH_CHECK();
    }
    return PSOAP_OK;
}

int fill_value(double* p, int64_t n, double v, cudaStream_t st) {
    if (n <= 0 || !p) return PSOAP_OK;
    grad_fill_kernel<<<(unsigned)std::min<int64_t>((n + 255) / 256, 1024), 256, 0, st>>>(p, n, v);
    LAUNCH_CHECK();
    return PSOAP_OK;
}
}  // namespace

extern "C" size_t psoap_lnlike_grad_workspace_bytes(int ncomp, int64_t N) {
    if (ncomp < 1 || ncomp > 3 || N < 0) return 0;
    GradWs g;
    return carve_grad_ws(nullptr, ncomp, N, 0, 0, &g);
}

extern "C" int psoap_lnlike_grad(int ncomp, int64_t N, const double* lwl_f, const double* lwl_g, const double* lwl_h,
                                 const double* fl, const double* sigma, const double* amp, const double* l, double mu_GP,
                                 void* workspace, size_t workspace_bytes, psoap_result* result, double* grad_hyp,
                                 double* grad_lwl, void* stream) {
    if (ncomp < 1 || ncomp > 3 || N < 0 || N > 200000 || !amp || !l || !result || !grad_hyp)
        return fail(PSOAP_ERR_ARG, "psoap_lnlike_grad: bad arguments");
    cudaStream_t st = (cudaStream_t)stream;
    const int nh = 2 * ncomp + 1;
    GpParams gp;
    if (make_gp(ncomp, amp, l, &gp)) {  // negative hyper-parameters: -inf, and no gradient
        write_result_kernel<<<1, 1, 0, st>>>((double*)result, -INFINITY, 0.0, 0.0, 0.0);
        LAUNCH_CHECK();
        int rc = fill_value(grad_hyp, nh, NAN, st);
        if (!rc) rc = fill_value(grad_lwl, (int64_t)ncomp * N, NAN, st);
        return rc;
    }
    if (N == 0) {  // empty chunk: -0.0 (see psoap_lnlike), nothing depends on the parameters
        write_result_kernel<<<1, 1, 0, st>>>((double*)result, -0.0, 0.0, 0.0, 0.0);
        LAUNCH_CHECK();
        return fill_value(grad_hyp, nh, 0.0, st);
    }
    if (!lwl_f || (ncomp > 1 && !lwl_g) || (ncomp > 2 && !lwl_h) || !fl || !sigma)
        return fail(PSOAP_ERR_ARG, "psoap_lnlike_grad: null vector");
    if (!workspace || workspace_bytes < psoap_lnlike_grad_workspace_bytes(ncomp, N) || ((uintptr_t)workspace & 255))
        return fail(PSOAP_ERR_WORKSPACE, "psoap_lnlike_grad: workspace too small or not 256-byte aligned");
    int rc = set_kernel_attributes();
    if (rc) return rc;
    GradWs g;
    carve_grad_ws((char*)workspace, ncomp, N, 0, 0, &g);
    Lanes ln;
    rc = get_lanes(st, &ln);
    if (rc) return rc;
    return launch_grad(ln, ncomp, N, direct_z(lwl_f, lwl_g, lwl_h), fl, sigma, mu_GP, gp, g, nullptr, (double*)result,
                       grad_hyp, grad_lwl);
}

extern "C" int psoap_lnlike_grad_views(void* workspace, int64_t N, double** neg_kinv_dev, int64_t* ld,
                                       double** neg_alpha_dev) {
    if (!workspace || N < 0) return fail(PSOAP_ERR_ARG, "psoap_lnlike_grad_views: bad arguments");
    GradWs g;
    carve_grad_ws((char*)workspace, 1, N, 0, 0, &g);
    if (neg_kinv_dev) *neg_kinv_dev = g.S + g.Nn + g.Nn * g.Nt;
    if (ld) *ld = g.Nt;
    if (neg_alpha_dev) *neg_alpha_dev = g.f.rvec + g.Nn;
    return PSOAP_OK;
}

extern "C" size_t psoap_chunk_lnprob_grad_workspace_bytes(int model, int64_t N, int32_t n_epochs) {
    if (model < 1 || model > 5 || N < 1 || n_epochs < 1) return 0;
    GradWs g;
    return carve_grad_ws(nullptr, model_ncomp(model), N, n_epochs, model_norb(model), &g);
}

namespace {
// the per-epoch sums and the chain rule of one gradient problem (the last steps of psoap_chunk_lnprob_grad)
int launch_grad_chain(cudaStream_t st, int ncomp, int norb, const psoap_chunk& ch, const GradWs& w, const double* jac,
                      const int* sentinel, double* grad_p) {
    grad_epoch_kernel<<<(unsigned)(ncomp * ch.n_epochs), 256, 0, st>>>(w.gz, ch.epoch, ch.N, ch.n_epochs, w.gv);
    LAUNCH_CHECK();
    grad_chain_kernel<<<1, 32, 0, st>>>(w.gv, jac, w.hyp, ncomp, ch.n_epochs, norb, w.f.info, sentinel, grad_p);
    LAUNCH_CHECK();
    return PSOAP_OK;
}

// The launches of psoap_chunk_lnprob_grad on a carved workspace: orbit velocities and sentinel, fill, identity border,
// restricted elimination, contraction, reductions, orbit Jacobian, per-epoch sum and chain rule.
int launch_chunk_grad(int model, const psoap_chunk* chunk, const double* p_dev, double mu_GP, const GradWs& g,
                      cudaStream_t st, double* result, double* grad_p) {
    const int ne = chunk->n_epochs, ncomp = model_ncomp(model), norb = model_norb(model);
    // orbit velocities and the sentinel (|v| >= c, or a negative GP hyper-parameter), as the farm's orbit kernel
    orbit_kernel<<<1, 128, 0, st>>>(model, p_dev, chunk->dates, ne, g.vel, g.flag, 1);
    LAUNCH_CHECK();
    Lanes ln;
    int rc = get_lanes(st, &ln);
    if (rc) return rc;
    rc = launch_grad(ln, ncomp, chunk->N, farm_z(*chunk, g.vel), chunk->fl, chunk->sigma, mu_GP, gp_params(p_dev + norb),
                     g, g.flag, result, g.hyp, g.gz);
    if (rc) return rc;
    orbit_jacobian_kernel<<<1, 128, 0, st>>>(model, p_dev, chunk->dates, ne, g.jac);
    LAUNCH_CHECK();
    return launch_grad_chain(st, ncomp, norb, *chunk, g, g.jac, g.flag, grad_p);
}

bool chunk_args_ok(int model, const psoap_chunk* chunk) {
    return model >= 1 && model <= 5 && chunk && chunk->N >= 1 && chunk->N <= 200000 && chunk->n_epochs >= 1 &&
           chunk->lwl && chunk->epoch && chunk->fl && chunk->sigma && chunk->dates;
}
}  // namespace

extern "C" int psoap_chunk_lnprob_grad(int model, const psoap_chunk* chunk, const double* p_dev, double mu_GP,
                                       void* workspace, size_t workspace_bytes, psoap_result* result, double* grad_p,
                                       void* stream) {
    if (!chunk_args_ok(model, chunk) || !p_dev || !result || !grad_p)
        return fail(PSOAP_ERR_ARG, "psoap_chunk_lnprob_grad: bad arguments");
    const int64_t N = chunk->N;
    const int ne = chunk->n_epochs, ncomp = model_ncomp(model), norb = model_norb(model);
    if (!workspace || workspace_bytes < psoap_chunk_lnprob_grad_workspace_bytes(model, N, ne) ||
        ((uintptr_t)workspace & 255))
        return fail(PSOAP_ERR_WORKSPACE, "psoap_chunk_lnprob_grad: workspace too small or not 256-byte aligned");
    int rc = set_kernel_attributes();
    if (rc) return rc;
    GradWs g;
    carve_grad_ws((char*)workspace, ncomp, N, ne, norb, &g);
    return launch_chunk_grad(model, chunk, p_dev, mu_GP, g, (cudaStream_t)stream, (double*)result, grad_p);
}

// ---- Fisher information of one chunk (fisher.cuh) ---------------------------------------------------------------
namespace {
// After the chunk's gradient workspace: the tile flags, the k ranges, the contraction partials, a gradient row for
// callers that want none, and the P products A_a = K^-1 D_a (the only O(N^2) addition: P Nn^2 doubles).
struct FisherWs {
    uint8_t* flags;   // [Tb][Tb]
    int* krange;      // [Tb][2]
    double* part;     // [Tb (Tb + 1) / 2][P (P + 1) / 2]
    double* grad_p;   // [P]
    double* prod;     // [P][Nn][Nn]
    int P, npairs;
};
size_t carve_fisher_ws(char* base, int model, int64_t N, int n_epochs, GradWs* g, FisherWs* f) {
    const int ncomp = model_ncomp(model), norb = model_norb(model);
    size_t off = carve_grad_ws(base, ncomp, N, n_epochs, norb, g);
    auto take = [&](size_t bytes) { char* r = base ? base + off : nullptr; off += align_up(bytes, 256); return r; };
    const int64_t Tb = g->Tb;
    f->P = norb + 2 * ncomp;
    f->npairs = (int)(Tb * (Tb + 1) / 2);
    f->flags = (uint8_t*)take((size_t)(Tb * Tb));
    f->krange = (int*)take((size_t)Tb * 2 * 4);
    f->part = (double*)take((size_t)f->npairs * (f->P * (f->P + 1) / 2) * 8);
    f->grad_p = (double*)take((size_t)f->P * 8);
    f->prod = (double*)take((size_t)f->P * g->Nn * g->Nn * 8);
    return off;
}

// the Fisher steps after launch_chunk_grad (fisher.cuh): mirror K^-1, then per parameter D_a and A_a = K^-1 D_a, then
// the tile-pair contraction and the fixed-order reduction into fisher [P][P]
int launch_fisher(int model, const psoap_chunk* chunk, const double* p_dev, const GradWs& g, const FisherWs& f,
                  cudaStream_t st, double* fisher) {
    const int N = (int)chunk->N, ncomp = model_ncomp(model), norb = model_norb(model), P = f.P;
    const int64_t Nn = g.Nn;
    double* kinv = g.S + Nn + Nn * g.Nt;
    const int T32 = (int)(Nn / 32);
    fisher_mirror_kernel<<<(unsigned)((int64_t)T32 * (T32 + 1) / 2), 256, 0, st>>>(kinv, g.Nt, N);
    LAUNCH_CHECK();
    CUtensorMap mapS, mapD;
    int rc = make_tensor_map(&mapS, kinv, (uint64_t)Nn, (uint64_t)Nn, (uint64_t)g.Nt, SA);
    if (!rc) rc = make_tensor_map(&mapD, g.S, (uint64_t)Nn, (uint64_t)Nn, (uint64_t)g.Nt, SB);
    if (rc) return rc;
    const ZSource zs = farm_z(*chunk, g.vel);
    const GpParams gp = gp_params(p_dev + norb);
    const int ntiles = g.Tb * 2 * g.Tb;
    for (int a = 0; a < P; ++a) {
        uint8_t* flags = (a == 0) ? f.flags : nullptr;   // the zero pattern is the same for every parameter
        with_ncomp(ncomp, [&](auto nc) {
            fisher_dk_kernel<nc><<<(unsigned)(g.Tb * g.Tb), 256, 0, st>>>(g.S, g.Nt, g.Tb, N, zs, gp, g.jac, norb, a, flags);
        });
        LAUNCH_CHECK();
        if (a == 0) {
            fisher_krange_kernel<<<1, 256, 0, st>>>(f.flags, g.Tb, f.krange);
            LAUNCH_CHECK();
        }
        FisherSrc src;
        src.krange = f.krange; src.C = f.prod + (int64_t)a * Nn * Nn; src.ldc = Nn; src.Tb = g.Tb;
        fisher_gemm_kernel<<<persistent_ctas(ntiles), 256, GEMM_SMEM, st>>>(src, ntiles, mapS, mapD);
        LAUNCH_CHECK();
    }
    fisher_pair_kernel<<<(unsigned)f.npairs, 256, fisher_pair_smem(P), st>>>(f.prod, Nn * Nn, Nn, P, f.part);
    LAUNCH_CHECK();
    fisher_reduce_kernel<<<1, 256, 0, st>>>(f.part, f.npairs, P, g.f.info, g.flag, fisher);
    LAUNCH_CHECK();
    return PSOAP_OK;
}
}  // namespace

extern "C" size_t psoap_chunk_fisher_workspace_bytes(int model, int64_t N, int32_t n_epochs) {
    if (model < 1 || model > 5 || N < 1 || N > 200000 || n_epochs < 1) return 0;
    GradWs g;
    FisherWs f;
    return carve_fisher_ws(nullptr, model, N, n_epochs, &g, &f);
}

extern "C" int psoap_chunk_fisher(int model, const psoap_chunk* chunk, const double* p_dev, double mu_GP,
                                  void* workspace, size_t workspace_bytes, psoap_result* result, double* grad_p,
                                  double* fisher, void* stream) {
    if (!chunk_args_ok(model, chunk) || !p_dev || !result || !fisher)
        return fail(PSOAP_ERR_ARG, "psoap_chunk_fisher: bad arguments");
    if (!workspace || workspace_bytes < psoap_chunk_fisher_workspace_bytes(model, chunk->N, chunk->n_epochs) ||
        ((uintptr_t)workspace & 255))
        return fail(PSOAP_ERR_WORKSPACE, "psoap_chunk_fisher: workspace too small or not 256-byte aligned");
    int rc = set_kernel_attributes();
    if (rc) return rc;
    GradWs g;
    FisherWs f;
    carve_fisher_ws((char*)workspace, model, chunk->N, chunk->n_epochs, &g, &f);
    const cudaStream_t st = (cudaStream_t)stream;
    rc = launch_chunk_grad(model, chunk, p_dev, mu_GP, g, st, (double*)result, grad_p ? grad_p : f.grad_p);
    if (rc) return rc;
    return launch_fisher(model, chunk, p_dev, g, f, st, fisher);
}

extern "C" int psoap_chunk_fisher_views(void* workspace, int model, int64_t N, int32_t n_epochs, uint8_t** flags,
                                        int** krange, int* Tb) {
    if (!workspace || model < 1 || model > 5 || N < 1 || n_epochs < 1)
        return fail(PSOAP_ERR_ARG, "psoap_chunk_fisher_views: bad arguments");
    GradWs g;
    FisherWs f;
    carve_fisher_ws((char*)workspace, model, N, n_epochs, &g, &f);
    if (flags) *flags = f.flags;
    if (krange) *krange = f.krange;
    if (Tb) *Tb = g.Tb;
    return PSOAP_OK;
}

extern "C" int psoap_orbit_jacobian(int model, const double* p_orb_dev, const double* dates_dev, int n_epochs,
                                    double* jac_dev, void* stream) {
    if (model < 1 || model > 5 || !p_orb_dev || !dates_dev || !jac_dev || n_epochs < 0)
        return fail(PSOAP_ERR_ARG, "psoap_orbit_jacobian: bad arguments");
    if (n_epochs == 0) return PSOAP_OK;
    orbit_jacobian_kernel<<<1, 128, 0, (cudaStream_t)stream>>>(model, p_orb_dev, dates_dev, n_epochs, jac_dev);
    LAUNCH_CHECK();
    return PSOAP_OK;
}

// ---- prediction as ONE entry (psoap/covariance.py:25-297) ----------------------------------------------
namespace {
int predict_dims(int ncomp, int mode, int64_t n, int64_t m, int64_t* M, int64_t* Nn, int64_t* Nt) {
    if (ncomp < 1 || ncomp > 3 || mode < 0 || mode > 2 || n < 1 || m < 1 || n > 200000 || m > 200000) return 1;
    if (mode == 2 && m != n) return 1;
    *M = (mode == 0) ? ncomp * m : m;
    *Nn = padded_dim(n);
    *Nt = *Nn + padded_dim(*M);
    return 0;
}
}  // namespace

extern "C" size_t psoap_predict_workspace_bytes(int ncomp, int mode, int64_t n, int64_t m) {
    int64_t M, Nn, Nt;
    if (predict_dims(ncomp, mode, n, m, &M, &Nn, &Nt)) return 0;
    return align_up((size_t)Nt * Nt * 8, 256) + psoap_schur_workspace_bytes(n, M);
}

extern "C" int psoap_predict(int ncomp, int mode, int64_t n, int64_t m, const double* const* lwl_data,
                             const double* fl, const double* sigma, const double* const* lwl_predict, const double* amp,
                             const double* l, double resid_mu, double nugget, double* delta_out, double* Sigma_out,
                             void* workspace, size_t workspace_bytes, psoap_result* result, void* stream) {
    int64_t M, Nn, Nt;
    if (predict_dims(ncomp, mode, n, m, &M, &Nn, &Nt) || !lwl_data || !fl || !sigma || !lwl_predict || !amp || !l ||
        !delta_out || !result)
        return fail(PSOAP_ERR_ARG, "psoap_predict: bad arguments");
    for (int c = 0; c < ncomp; ++c)
        if (!lwl_data[c] || !lwl_predict[c]) return fail(PSOAP_ERR_ARG, "psoap_predict: null vector");
    if (!workspace || workspace_bytes < psoap_predict_workspace_bytes(ncomp, mode, n, m) || ((uintptr_t)workspace & 255))
        return fail(PSOAP_ERR_WORKSPACE, "psoap_predict: workspace too small or not 256-byte aligned");
    int rc = set_kernel_attributes();
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    double* S = (double*)workspace;
    FactorWs ws;
    carve_factor_ws((char*)workspace + align_up((size_t)Nt * Nt * 8, 256), Nt, &ws, false);
    GpParams gp;
    make_gp(ncomp, amp, l, &gp);
    const int pad = (int)(Nn - n);
    // data block: the likelihood's own fill (lower triangle, front padding, residual fl - resid_mu, accumulator reset)
    rc = launch_fill_lower(ncomp, st, S, Nt, (int)(Nn / NB), pad, direct_z(lwl_data[0], ncomp > 1 ? lwl_data[1] : nullptr,
                                                                          ncomp > 2 ? lwl_data[2] : nullptr),
                           sigma, fl, resid_mu, gp, ws);
    if (rc) return rc;
    PredictSrc ps;
    for (int c = 0; c < 3; ++c) { ps.data[c] = c < ncomp ? lwl_data[c] : nullptr; ps.pred[c] = c < ncomp ? lwl_predict[c] : nullptr; }
    ps.ncomp = ncomp; ps.mode = mode; ps.n = (int)n; ps.m = (int)m; ps.M = (int)M;
    ps.pad = pad; ps.Nn = (int)Nn; ps.Nt = (int)Nt; ps.nugget = nugget;
    const int Tn = (int)(Nn / NB), Tt = (int)(Nt / NB);
    const unsigned ntile = (unsigned)((int64_t)Tt * (Tt + 1) / 2 - (int64_t)Tn * (Tn + 1) / 2);
    with_ncomp(ncomp, [&](auto nc) { predict_border_kernel<nc><<<ntile, 256, 0, st>>>(S, Nt, ps, gp, ws.rvec); });
    LAUNCH_CHECK();
    Lanes ln;
    rc = get_lanes(st, &ln);
    if (rc) return rc;
    rc = launch_factor(ln, S, Nt, Tn, Tt, pad, ws, nullptr, (double*)result);
    if (rc) return rc;
    const unsigned nb = (unsigned)((M + 31) / 32);
    predict_readout_kernel<<<dim3(nb, nb), 256, 0, st>>>(S, Nt, (int)Nn, (int)M, ws.rvec, Sigma_out, delta_out);
    LAUNCH_CHECK();
    return PSOAP_OK;
}

// Host buffers in, host buffers out (synchronous): what a C caller without device memory binds.
extern "C" int psoap_predict_host(int ncomp, int mode, int64_t n, int64_t m, const double* const* lwl_data,
                                  const double* fl, const double* sigma, const double* const* lwl_predict,
                                  const double* amp, const double* l, double resid_mu, double nugget,
                                  double* delta_out, double* Sigma_out, psoap_result* result) {
    int64_t M, Nn, Nt;
    if (predict_dims(ncomp, mode, n, m, &M, &Nn, &Nt) || !lwl_data || !fl || !sigma || !lwl_predict || !amp || !l ||
        !delta_out || !result)
        return fail(PSOAP_ERR_ARG, "psoap_predict_host: bad arguments");
    for (int c = 0; c < ncomp; ++c)
        if (!lwl_data[c] || !lwl_predict[c]) return fail(PSOAP_ERR_ARG, "psoap_predict_host: null vector");
    const size_t wsb = psoap_predict_workspace_bytes(ncomp, mode, n, m);
    const size_t vn = align_up((size_t)n * 8, 256), vm = align_up((size_t)m * 8, 256), vM = align_up((size_t)M * 8, 256);
    const size_t sig = Sigma_out ? align_up((size_t)M * M * 8, 256) : 0;
    const size_t total = wsb + (size_t)(ncomp + 2) * vn + (size_t)ncomp * vm + vM + sig + 512;
    char* base = nullptr;
    CUDA_TRY(cudaMalloc(&base, total));
    cudaStream_t st = nullptr;
    cudaError_t e = cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking);
    int rc = PSOAP_OK;
    if (e == cudaSuccess) {
        char* p = base + wsb;
        auto take = [&](size_t b) { char* r = p; p += b; return (double*)r; };
        const double *dd[3] = {nullptr, nullptr, nullptr}, *dp[3] = {nullptr, nullptr, nullptr};
        for (int c = 0; c < ncomp && e == cudaSuccess; ++c) {
            double* x = take(vn); dd[c] = x;
            e = cudaMemcpyAsync(x, lwl_data[c], (size_t)n * 8, cudaMemcpyHostToDevice, st);
            double* y = take(vm); dp[c] = y;
            if (e == cudaSuccess) e = cudaMemcpyAsync(y, lwl_predict[c], (size_t)m * 8, cudaMemcpyHostToDevice, st);
        }
        double* dfl = take(vn); double* dsg = take(vn); double* ddelta = take(vM);
        double* dSig = Sigma_out ? take(sig) : nullptr;
        psoap_result* dres = (psoap_result*)take(256);
        if (e == cudaSuccess) e = cudaMemcpyAsync(dfl, fl, (size_t)n * 8, cudaMemcpyHostToDevice, st);
        if (e == cudaSuccess) e = cudaMemcpyAsync(dsg, sigma, (size_t)n * 8, cudaMemcpyHostToDevice, st);
        if (e == cudaSuccess)
            rc = psoap_predict(ncomp, mode, n, m, dd, dfl, dsg, dp, amp, l, resid_mu, nugget, ddelta, dSig, base, wsb, dres, st);
        if (e == cudaSuccess && rc == PSOAP_OK) {
            e = cudaMemcpyAsync(delta_out, ddelta, (size_t)M * 8, cudaMemcpyDeviceToHost, st);
            if (e == cudaSuccess && Sigma_out) e = cudaMemcpyAsync(Sigma_out, dSig, (size_t)M * M * 8, cudaMemcpyDeviceToHost, st);
            if (e == cudaSuccess) e = cudaMemcpyAsync(result, dres, sizeof(psoap_result), cudaMemcpyDeviceToHost, st);
        }
        cudaError_t e2 = cudaStreamSynchronize(st);
        if (e == cudaSuccess) e = e2;
        cudaStreamDestroy(st);
    }
    cudaFree(base);
    if (rc) return rc;
    if (e != cudaSuccess) return fail(PSOAP_ERR_CUDA, std::string("psoap_predict_host: ") + cudaGetErrorString(e));
    return PSOAP_OK;
}

// ======================================================================================================
// Chunk farm
// ======================================================================================================
constexpr int P_STRIDE = 32;  // doubles reserved per proposal in the parameter buffer
namespace {
// One CUDA graph of a farm: the state of its work items (item = proposal * nchunks + chunk), the branch scratch, and
// what issues it: the branch streams (+ the root stream at index nbranch), their events, the high-priority side streams
// of look-ahead, and whether calls replay the captured graph or issue the kernels directly.  The likelihood graph, the
// gradient graph and the prediction graph each own one; it releases its streams, events and graph with it.
struct FarmGraph {
    int nbranch = 0;
    bool lookahead = false;
    bool direct = false;              // issue the kernels on every call instead of replaying the captured graph
    cudaGraph_t graph = nullptr;
    cudaGraphExec_t exec = nullptr;
    std::vector<cudaStream_t> streams;
    std::vector<cudaStream_t> side_streams;
    std::vector<cudaEvent_t> events;
    std::vector<cudaEvent_t> side_events;
    int launches = 0;                 // kernels one evaluation launches
    double* p_buf = nullptr;          // [nprop][P_STRIDE] parameter vectors the graph reads
    double* results = nullptr;        // [nitems][4]
    int* flags = nullptr;             // per item sentinel
    OrbitDesc* descs = nullptr;       // device, per item
    std::vector<double*> item_vel;    // device velocity table of each item
    std::vector<char*> branch_base;   // scratch region of each branch, carved for each of its items in turn (items of
                                      // a branch run in stream order)
    std::vector<std::vector<int>> branch_items;   // LPT order

    FarmGraph() = default;
    FarmGraph(const FarmGraph&) = delete;
    FarmGraph& operator=(const FarmGraph&) = delete;
    ~FarmGraph() {
        if (exec) cudaGraphExecDestroy(exec);
        if (graph) cudaGraphDestroy(graph);
        for (auto& s : streams) if (s) cudaStreamDestroy(s);
        for (auto& s : side_streams) if (s) cudaStreamDestroy(s);
        for (auto& ev : events) if (ev) cudaEventDestroy(ev);
        for (auto& ev : side_events) if (ev) cudaEventDestroy(ev);
    }
};

// The optional gradient graph of a farm (psoap_farm_grad_attach): besides the item state, the gradient rows and orbit
// Jacobians of every item.  Each branch region holds one GradWs.
struct FarmGrad {
    FarmGraph g;
    double* grad = nullptr;           // [nitems][n_params]
    JacDesc* jdescs = nullptr;        // device, per item
    std::vector<double*> item_jac;    // [ncomp][n_epochs][norb] per item
};

// The optional prediction graph of a farm (psoap_farm_predict_attach): besides the item state, the caller's grids and
// the output offsets of every item.  Each branch region holds the bordered matrix of an item (S, then its FactorWs).
struct FarmPredict {
    FarmGraph g;
    int sigma_mode = 0;               // 0: Sigma [M][M], 1: its diagonal [M]
    std::vector<int64_t> m;           // grid points per component, per chunk
    std::vector<const double*> grids; // [nchunks][ncomp] device pointers
    std::vector<int64_t> delta_off;   // [nitems + 1] offsets (doubles) into delta_dev; the last one is its length
    std::vector<int64_t> sigma_off;   // [nitems + 1] the same into sigma_dev
    double* cap_delta = nullptr;      // scratch outputs the captured graph writes; copied out after a replay
    double* cap_sigma = nullptr;
};
}  // namespace

struct psoap_farm {
    int model = 0, ncomp = 0, norb = 0, nchunks = 0, nprop = 1, nitems = 0;
    double mu = 1.0;
    std::vector<psoap_chunk> chunks;
    FarmGraph g;                      // the likelihood graph
    int chain_hint = 0;               // psoap_chunk.reserved of the first chunk, low byte: 3 | 7 forces the chain links
    int group_hint = 0;               // ... bits 8 and up: 2 | 4 | 8 forces the panels per trailing update
    FarmGrad* grad = nullptr;         // psoap_farm_grad_attach; null until then
    FarmPredict* pred = nullptr;      // psoap_farm_predict_attach; null until then
    ~psoap_farm() { delete grad; delete pred; }
};

namespace {
// The launch plan of one work item on branch b of graph g, shared by the likelihood, gradient and prediction graphs so
// that they cannot drift apart.
Lanes farm_lanes(const psoap_farm* f, const FarmGraph& g, int b, int pdl) {
    Lanes ln;
    ln.main = g.streams[b];
    ln.side = g.lookahead ? g.side_streams[b] : nullptr;
    ln.e1 = g.side_events[2 * b]; ln.e2 = g.side_events[2 * b + 1];
    // panels per update: the caller's choice (bits 8.. of psoap_chunk.reserved: 2, 4 or 8, again the same on every
    // rank), else by the number of chunks in flight: rank-1024 updates need many to hide their 8-panel heads (C1
    // x 8 proposals on 8 branches: 1121 evals/s against 1149 with rank-512)
    ln.group = g.lookahead ? 0
             : (f->group_hint == 2 || f->group_hint == 4 || f->group_hint == 8) ? f->group_hint
             : (g.nbranch >= 32 ? 8 : 4);
    ln.pdl = pdl;
    // chain links: the caller's choice (psoap_chunk.reserved = 3 | 7, the same on every rank of a partitioned
    // farm so that the bits do not depend on the number of GPUs), else by exposure of the chain latency
    ln.chain = (f->chain_hint == 3 || f->chain_hint == 7) ? f->chain_hint : (g.lookahead ? 0 : 3);
    return ln;
}

// the GP values of item it's proposal, as every farm graph reads them
GpParams farm_gp(const psoap_farm* f, const FarmGraph& g, int it) {
    return gp_params(g.p_buf + (size_t)(it / f->nchunks) * P_STRIDE + f->norb);
}

// Forks g's branches from s0, after the root kernels the caller launched there, issues the items of each branch in LPT
// order through item(b, branch stream, it), and joins the branches back into s0.
template <class Item>
int issue_branches(const FarmGraph& g, cudaStream_t s0, Item&& item) {
    const cudaEvent_t fork = g.events[g.nbranch];
    CUDA_TRY(cudaEventRecord(fork, s0));
    int rc = PSOAP_OK;
    for (int b = 0; b < g.nbranch && rc == PSOAP_OK; ++b) {
        const cudaStream_t sb = g.streams[b];
        CUDA_TRY(cudaStreamWaitEvent(sb, fork, 0));
        for (int it : g.branch_items[b])
            if ((rc = item(b, sb, it)) != PSOAP_OK) break;
        CUDA_TRY(cudaEventRecord(g.events[b], sb));
        CUDA_TRY(cudaStreamWaitEvent(s0, g.events[b], 0));
    }
    return rc;
}

// Issues one evaluation onto the likelihood graph's streams, rooted at s0: the orbit kernel for every item, then the
// per-chunk pipelines on the branch streams.  Runs under stream capture (graph mode) or for real (direct mode, which
// adds programmatic dependent launch on the small grids).
int farm_issue(const psoap_farm* f, cudaStream_t s0, int pdl) {
    const FarmGraph& g = f->g;
    orbit_farm_kernel<<<f->nitems, 64, 0, s0>>>(f->model, g.p_buf, g.descs);
    LAUNCH_CHECK();
    return issue_branches(g, s0, [&](int b, cudaStream_t, int it) {
        const psoap_chunk& ch = f->chunks[it % f->nchunks];
        FactorWs ws;
        carve_factor_ws(g.branch_base[b], padded_dim(ch.N), &ws, true);
        return launch_chunk(farm_lanes(f, g, b, pdl), f->ncomp, ch.N, farm_z(ch, g.item_vel[it]), ch.fl, ch.sigma, f->mu,
                            farm_gp(f, g, it), ws, g.flags + it, g.results + 4 * it);
    });
}

// The gradient counterpart of farm_issue: velocities, sentinels and orbit Jacobians of every item, then per branch the
// steps of psoap_chunk_lnprob_grad into the item's result and gradient rows.
int farm_grad_issue(const psoap_farm* f, const FarmGrad& q, cudaStream_t s0, int pdl) {
    const FarmGraph& g = q.g;
    const int np = f->norb + 2 * f->ncomp;
    orbit_farm_kernel<<<f->nitems, 64, 0, s0>>>(f->model, g.p_buf, g.descs);
    LAUNCH_CHECK();
    orbit_jacobian_farm_kernel<<<f->nitems, 64, 0, s0>>>(f->model, g.p_buf, q.jdescs);
    LAUNCH_CHECK();
    return issue_branches(g, s0, [&](int b, cudaStream_t sb, int it) {
        const psoap_chunk& ch = f->chunks[it % f->nchunks];
        GradWs w;
        carve_grad_ws(g.branch_base[b], f->ncomp, ch.N, ch.n_epochs, f->norb, &w);
        int rc = launch_grad(farm_lanes(f, g, b, pdl), f->ncomp, ch.N, farm_z(ch, g.item_vel[it]), ch.fl, ch.sigma, f->mu,
                             farm_gp(f, g, it), w, g.flags + it, g.results + 4 * it, w.hyp, w.gz);
        if (!rc) rc = launch_grad_chain(sb, f->ncomp, f->norb, ch, w, q.item_jac[it], g.flags + it, q.grad + (size_t)it * np);
        return rc;
    });
}

// Bordered dimensions of one prediction item: data block Nn (front-padded), border M = ncomp m, total Nt.
struct PredictDims { int64_t Nn, M, Nt; };
PredictDims predict_item_dims(int ncomp, int64_t N, int64_t m) {
    const int64_t Nn = padded_dim(N), M = ncomp * m;
    return {Nn, M, Nn + padded_dim(M)};
}

// The prediction counterpart of farm_issue: velocities and sentinels of every item, then per branch the steps of
// psoap_predict (mode 0) on the item's shifted pixels: data fill, border fill, elimination of the data block, read-out
// into the item's offsets of delta and sigma.
int farm_predict_issue(const psoap_farm* f, const FarmPredict& q, cudaStream_t s0, int pdl, double* delta, double* sigma) {
    const FarmGraph& g = q.g;
    const int nchunks = f->nchunks, ncomp = f->ncomp;
    orbit_farm_kernel<<<f->nitems, 64, 0, s0>>>(f->model, g.p_buf, g.descs);
    LAUNCH_CHECK();
    return issue_branches(g, s0, [&](int b, cudaStream_t sb, int it) {
        const int ci = it % nchunks;
        const psoap_chunk& ch = f->chunks[ci];
        const PredictDims d = predict_item_dims(ncomp, ch.N, q.m[ci]);
        const int Tn = (int)(d.Nn / NB), Tt = (int)(d.Nt / NB), pad = (int)(d.Nn - ch.N);
        FactorWs ws;
        carve_factor_ws(g.branch_base[b], d.Nt, &ws, true);
        const GpParams gp = farm_gp(f, g, it);
        const ZSource zs = farm_z(ch, g.item_vel[it]);
        int rc = launch_fill_lower(ncomp, sb, ws.W, d.Nt, Tn, pad, zs, ch.sigma, ch.fl, f->mu, gp, ws);
        if (rc) return rc;
        PredictFarmSrc ps;
        for (int c = 0; c < 3; ++c) { ps.data[c] = nullptr; ps.pred[c] = c < ncomp ? q.grids[(size_t)ci * ncomp + c] : nullptr; }
        ps.ncomp = ncomp; ps.mode = 0; ps.n = (int)ch.N; ps.m = (int)q.m[ci]; ps.M = (int)d.M;
        ps.pad = pad; ps.Nn = (int)d.Nn; ps.Nt = (int)d.Nt; ps.nugget = 0.0; ps.zs = zs;
        const unsigned ntile = (unsigned)((int64_t)Tt * (Tt + 1) / 2 - (int64_t)Tn * (Tn + 1) / 2);
        with_ncomp(ncomp, [&](auto nc) {
            predict_border_farm_kernel<nc><<<ntile, 256, 0, sb>>>(ws.W, d.Nt, ps, gp, ws.rvec);
        });
        LAUNCH_CHECK();
        rc = launch_factor(farm_lanes(f, g, b, pdl), ws.W, d.Nt, Tn, Tt, pad, ws, g.flags + it, g.results + 4 * it);
        if (rc) return rc;
        const unsigned nb = (unsigned)((d.M + 31) / 32);
        predict_farm_readout_kernel<<<dim3(q.sigma_mode ? 1u : nb, nb), 256, 0, sb>>>(
            ws.W, d.Nt, (int)d.Nn, (int)d.M, ws.rvec, ws.info, g.flags + it, q.sigma_mode, sigma + q.sigma_off[it],
            delta + q.delta_off[it]);
        LAUNCH_CHECK();
        return PSOAP_OK;
    });
}

// LPT (longest processing time first) assignment of work items (item = prop * nchunks + chunk) to branches by N^3;
// items of chunks with N = 0 are left out
std::vector<std::vector<int>> lpt_items(const std::vector<int64_t>& Ns, int nitems, int nbranch) {
    const int nchunks = (int)Ns.size();
    std::vector<int> order;
    for (int it = 0; it < nitems; ++it)
        if (Ns[it % nchunks] > 0) order.push_back(it);
    std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return Ns[a % nchunks] > Ns[b % nchunks]; });
    std::vector<double> load(nbranch, 0.0);
    std::vector<std::vector<int>> items(nbranch);
    for (int it : order) {
        int b = (int)(std::min_element(load.begin(), load.end()) - load.begin());
        items[b].push_back(it);
        const double n = (double)Ns[it % nchunks];
        load[b] += n * n * n;
    }
    return items;
}

// Branch streams (+ the root stream at index nbranch), their events, and the high-priority side streams of look-ahead
int create_farm_streams(FarmGraph& g) {
    const int nbranch = g.nbranch;
    g.streams.resize(nbranch + 1);
    g.events.resize(nbranch + 1);
    g.side_streams.resize(nbranch);
    g.side_events.resize(2 * nbranch);
    int lo = 0, hi = 0;
    CUDA_TRY(cudaDeviceGetStreamPriorityRange(&lo, &hi));
    // Branch b carries the b-th largest items first (LPT order): its stream gets the matching priority level, which a
    // captured kernel node inherits.  Measured neutral on a B200 against all-equal priorities (one rank's share of
    // an 8-GPU run: 28.50 ms either way; a launch-attribute variant likewise): the drain at the end of an evaluation
    // is not a matter of which chunk gets the free SM slots first.
    const int nlev = lo - hi + 1;
    for (int b = 0; b <= nbranch; ++b) {
        // (a look-ahead farm's branch streams carry the bulk updates: lowest priority, below their side streams, where
        // the chain links run; with both at the top C2 ran at 95.5 instead of 104 evals/s)
        const int pr = (b < nbranch && nlev > 1 && !g.lookahead) ? hi + (int)((int64_t)b * nlev / nbranch) : lo;
        CUDA_TRY(cudaStreamCreateWithPriority(&g.streams[b], cudaStreamNonBlocking, pr));
    }
    for (auto& s : g.side_streams) CUDA_TRY(cudaStreamCreateWithPriority(&s, cudaStreamNonBlocking, hi));
    for (auto& ev : g.events) CUDA_TRY(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
    for (auto& ev : g.side_events) CUDA_TRY(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
    return PSOAP_OK;
}

using FarmIssue = std::function<int(cudaStream_t s0, int pdl)>;

// Captures one evaluation, issued by `issue` onto g's streams, into g's graph and instantiates it.  The launches it
// counts are g.launches (capture is not execution: the library's launch counter is left as it was).
int capture_farm_graph(FarmGraph& g, const FarmIssue& issue) {
    cudaStream_t s0 = g.streams[g.nbranch];
    const int64_t before = g_launches.load();
    cudaError_t e = cudaStreamBeginCapture(s0, cudaStreamCaptureModeThreadLocal);
    if (e != cudaSuccess) return fail(PSOAP_ERR_CUDA, std::string("begin capture: ") + cudaGetErrorString(e));
    int rc = issue(s0, 0);
    e = cudaStreamEndCapture(s0, &g.graph);
    g.launches = (int)(g_launches.load() - before);
    g_launches = before;
    if (rc != PSOAP_OK) return rc;
    if (e != cudaSuccess) return fail(PSOAP_ERR_CUDA, std::string("end capture: ") + cudaGetErrorString(e));
    e = cudaGraphInstantiate(&g.exec, g.graph, 0);
    if (e != cudaSuccess) return fail(PSOAP_ERR_CUDA, std::string("graph instantiate: ") + cudaGetErrorString(e));
    return PSOAP_OK;
}

// The setup of every farm graph once its workspace is carved: the orbit descriptors of its items, their LPT assignment
// to the branches by `cost` (per chunk, cubed by lpt_items; 0: no work), look-ahead and direct issue, the streams, and
// the capture.  On failure the caller deletes the graph's owner, which releases what was created.
int attach_farm_graph(const psoap_farm* f, FarmGraph& g, const std::vector<int64_t>& cost, bool attached,
                      const FarmIssue& issue) {
    std::vector<OrbitDesc> hd(f->nitems);
    for (int it = 0; it < f->nitems; ++it) {
        const psoap_chunk& ch = f->chunks[it % f->nchunks];
        hd[it] = {ch.dates, g.item_vel[it], g.flags + it, ch.n_epochs, (it / f->nchunks) * P_STRIDE};
    }
    CUDA_TRY(cudaMemcpy(g.descs, hd.data(), hd.size() * sizeof(OrbitDesc), cudaMemcpyHostToDevice));
    g.branch_items = lpt_items(cost, f->nitems, g.nbranch);
    int64_t nmax = 0;   // the largest chunk that takes work
    for (int i = 0; i < f->nchunks; ++i)
        if (cost[i] > 0) nmax = std::max(nmax, f->chunks[i].N);
    // Look-ahead changes the panel groups of the elimination, hence its bits.  When the caller passes the chain links
    // (psoap_chunk.reserved, chosen from the global problem: 7 for fewer than 8 (proposal, chunk) pairs in all), an
    // attached graph (gradient, prediction) takes look-ahead exactly there, so that its outputs depend neither on the
    // branch count nor on the number of GPUs; without that hint it decides by branch count.  The likelihood graph always
    // decides by branch count: taking the hint there would change the likelihood's bits on some partitioned farms.
    const char* la_env = getenv("PSOAP_FARM_LOOKAHEAD");
    const bool hinted = attached && (f->chain_hint == 3 || f->chain_hint == 7);
    g.lookahead = la_env ? (atoi(la_env) != 0) : hinted ? (f->chain_hint == 7) : (g.nbranch < 8);
    // Graph replay removes every launch gap, which wins for short chains (N = 4000: 2.57 vs 2.75 ms); for a farm of
    // a few LARGE chunks the directly issued pipeline is faster (N = 9000: 10.5 vs 11.3 ms: the side stream's
    // priority and the pre-staged small grids do their job there).  PSOAP_FARM_DIRECT=0|1 overrides.
    const char* de = getenv("PSOAP_FARM_DIRECT");
    g.direct = de ? (atoi(de) != 0) : (g.lookahead && nmax >= 7000);
    int rc = create_farm_streams(g);
    if (rc) return rc;
    return capture_farm_graph(g, issue);
}

// One evaluation of graph g at the parameters p_dev on the caller's stream st: the parameter upload, the captured
// graph's replay or (direct mode) the kernels issued on g's own streams, forked from st and joined back into it, and
// the copy of the result records.
int run_farm_graph(const psoap_farm* f, FarmGraph& g, const double* p_dev, psoap_result* results_dev, cudaStream_t st,
                   const FarmIssue& issue) {
    const int np = f->norb + 2 * f->ncomp;
    // p_dev: [nprop][np] contiguous -> [nprop][P_STRIDE]
    CUDA_TRY(cudaMemcpy2DAsync(g.p_buf, P_STRIDE * 8, p_dev, (size_t)np * 8, (size_t)np * 8, f->nprop,
                               cudaMemcpyDeviceToDevice, st));
    if (g.direct) {
        cudaStream_t s0 = g.streams[g.nbranch];
        cudaEvent_t fork = g.events[g.nbranch];
        CUDA_TRY(cudaEventRecord(fork, st));
        CUDA_TRY(cudaStreamWaitEvent(s0, fork, 0));
        int rc = issue(s0, g_pdl);
        if (rc) return rc;
        CUDA_TRY(cudaEventRecord(fork, s0));
        CUDA_TRY(cudaStreamWaitEvent(st, fork, 0));
    } else {
        CUDA_TRY(cudaGraphLaunch(g.exec, st));
        g_launches += g.launches;
    }
    CUDA_TRY(cudaMemcpyAsync(results_dev, g.results, (size_t)f->nitems * sizeof(psoap_result), cudaMemcpyDeviceToDevice, st));
    return PSOAP_OK;
}

// Bump allocation of 256-byte aligned pieces from base (null: offsets only, for the size queries)
struct Carver {
    char* base;
    size_t off = 0;
    char* take(size_t bytes) { char* r = base ? base + off : nullptr; off += align_up(bytes, 256); return r; }
};

// Layout of the part of a workspace every farm graph has: the parameter buffer, the result records, sentinels and orbit
// descriptors of the items, vel_rows x n_epochs velocity doubles per item, then nbranch regions of branch_bytes.  The
// graph's own buffers follow at c.off.
void carve_farm_items(Carver& c, FarmGraph& g, int nprop, int nchunks, const int32_t* n_epochs, int vel_rows,
                      size_t branch_bytes) {
    const int nitems = nchunks * nprop;
    g.p_buf = (double*)c.take((size_t)nprop * P_STRIDE * 8);
    g.results = (double*)c.take((size_t)nitems * 4 * 8);
    g.flags = (int*)c.take((size_t)nitems * 4);
    g.descs = (OrbitDesc*)c.take((size_t)nitems * sizeof(OrbitDesc));
    g.item_vel.resize(nitems);
    for (int it = 0; it < nitems; ++it) g.item_vel[it] = (double*)c.take((size_t)vel_rows * n_epochs[it % nchunks] * 8);
    g.branch_base.resize(g.nbranch);
    for (auto& r : g.branch_base) r = c.take(branch_bytes);
}

// Layout of a likelihood workspace: each branch holds the FactorWs of the largest chunk.  The size query takes no
// model, so every item reserves the velocity table of three components.
size_t carve_farm_lnprob(char* base, FarmGraph& g, int nchunks, const int64_t* N, const int32_t* n_epochs, int nprop) {
    int64_t nmax = 0;
    for (int i = 0; i < nchunks; ++i) nmax = std::max(nmax, N[i]);
    Carver c{base};
    carve_farm_items(c, g, nprop, nchunks, n_epochs, 3, factor_ws_bytes(padded_dim(nmax)));
    return c.off;
}

std::vector<int32_t> farm_epochs(const psoap_farm* f) {
    std::vector<int32_t> nes;
    for (const psoap_chunk& ch : f->chunks) nes.push_back(ch.n_epochs);
    return nes;
}

// Layout of a gradient workspace: each branch holds a GradWs sized for the largest chunk and the most epochs (every
// GradWs buffer grows with N and with n_epochs, so an item's carve fits), then the gradient rows, Jacobian descriptors
// and Jacobians of the items.
size_t carve_farm_grad(const psoap_farm* f, char* base, FarmGrad& q) {
    const int nitems = f->nitems, np = f->norb + 2 * f->ncomp;
    const std::vector<int32_t> nes = farm_epochs(f);
    int64_t nmax = 1;
    int nemax = 1;
    for (const psoap_chunk& ch : f->chunks) { nmax = std::max<int64_t>(nmax, ch.N); nemax = std::max(nemax, (int)ch.n_epochs); }
    GradWs probe;
    Carver c{base};
    carve_farm_items(c, q.g, f->nprop, f->nchunks, nes.data(), f->ncomp,
                     carve_grad_ws(nullptr, f->ncomp, nmax, nemax, f->norb, &probe));
    q.grad = (double*)c.take((size_t)nitems * np * 8);
    q.jdescs = (JacDesc*)c.take((size_t)nitems * sizeof(JacDesc));
    q.item_jac.resize(nitems);
    for (int it = 0; it < nitems; ++it) q.item_jac[it] = (double*)c.take((size_t)f->ncomp * nes[it % f->nchunks] * f->norb * 8);
    return c.off;
}

// Layout of a prediction workspace: each branch holds factor_ws_bytes(Nt) for the largest bordered item, then the
// graph's scratch outputs.  Also sets the output offsets of the items.
size_t carve_farm_predict(const psoap_farm* f, const int64_t* m, int sigma_mode, char* base, FarmPredict& q) {
    const int nitems = f->nitems, nchunks = f->nchunks;
    // output layout: chunk after chunk, each chunk's proposals side by side, so that a chunk's outputs are contiguous
    q.delta_off.resize(nitems + 1);
    q.sigma_off.resize(nitems + 1);
    int64_t nd = 0, ns = 0, ntmax = 0;
    for (int ci = 0; ci < nchunks; ++ci) {
        const PredictDims d = predict_item_dims(f->ncomp, f->chunks[ci].N, m[ci]);
        if (m[ci] > 0) ntmax = std::max(ntmax, d.Nt);
        for (int k = 0; k < f->nprop; ++k) {
            const int it = k * nchunks + ci;
            q.delta_off[it] = nd; q.sigma_off[it] = ns;
            nd += d.M; ns += sigma_mode ? d.M : d.M * d.M;
        }
    }
    q.delta_off[nitems] = nd; q.sigma_off[nitems] = ns;
    Carver c{base};
    carve_farm_items(c, q.g, f->nprop, nchunks, farm_epochs(f).data(), f->ncomp, ntmax ? factor_ws_bytes(ntmax) : 0);
    q.cap_delta = (double*)c.take((size_t)nd * 8);
    q.cap_sigma = (double*)c.take((size_t)ns * 8);
    return c.off;
}
}  // namespace

extern "C" {

size_t psoap_farm_workspace_bytes_batched(int nchunks, const int64_t* N, const int32_t* n_epochs, int nprop,
                                          int nbranch) {
    if (nchunks < 1 || nprop < 1 || !N || !n_epochs) return 0;
    FarmGraph probe;
    probe.nbranch = std::max(1, std::min(nbranch, nchunks * nprop));
    return carve_farm_lnprob(nullptr, probe, nchunks, N, n_epochs, nprop);
}
size_t psoap_farm_workspace_bytes(int nchunks, const int64_t* N, const int32_t* n_epochs, int nbranch) {
    return psoap_farm_workspace_bytes_batched(nchunks, N, n_epochs, 1, nbranch);
}

int psoap_farm_create_batched(psoap_farm** out, int model, int nchunks, const psoap_chunk* chunks, int nprop,
                              int nbranch, double mu_GP, void* workspace, size_t workspace_bytes) {
    if (!out || model < 1 || model > 5 || nchunks < 1 || nprop < 1 || !chunks || !workspace || ((uintptr_t)workspace & 255))
        return fail(PSOAP_ERR_ARG, "psoap_farm_create: bad arguments");
    const int nitems = nchunks * nprop;
    nbranch = std::max(1, std::min(nbranch, nitems));
    std::vector<int64_t> Ns(nchunks);
    std::vector<int32_t> nes(nchunks);
    for (int i = 0; i < nchunks; ++i) {
        if (chunks[i].N < 1 || chunks[i].n_epochs < 1 || !chunks[i].lwl || !chunks[i].epoch || !chunks[i].fl ||
            !chunks[i].sigma || !chunks[i].dates)
            return fail(PSOAP_ERR_ARG, "psoap_farm_create: bad chunk descriptor");
        Ns[i] = chunks[i].N;
        nes[i] = chunks[i].n_epochs;
    }
    if (workspace_bytes < psoap_farm_workspace_bytes_batched(nchunks, Ns.data(), nes.data(), nprop, nbranch))
        return fail(PSOAP_ERR_WORKSPACE, "psoap_farm_create: workspace too small");
    int rc = set_kernel_attributes();
    if (rc) return rc;

    psoap_farm* f = new psoap_farm();
    f->model = model; f->ncomp = model_ncomp(model); f->norb = model_norb(model);
    f->nchunks = nchunks; f->nprop = nprop; f->nitems = nitems; f->g.nbranch = nbranch; f->mu = mu_GP;
    f->chunks.assign(chunks, chunks + nchunks);
    f->chain_hint = chunks[0].reserved & 0xff;
    f->group_hint = (chunks[0].reserved >> 8) & 0xff;
    carve_farm_lnprob((char*)workspace, f->g, nchunks, Ns.data(), nes.data(), nprop);
    rc = attach_farm_graph(f, f->g, Ns, false, [f](cudaStream_t s0, int pdl) { return farm_issue(f, s0, pdl); });
    if (rc != PSOAP_OK) { delete f; return rc; }
    *out = f;
    return PSOAP_OK;
}

int psoap_farm_create(psoap_farm** out, int model, int nchunks, const psoap_chunk* chunks, int nbranch, double mu_GP,
                      void* workspace, size_t workspace_bytes) {
    return psoap_farm_create_batched(out, model, nchunks, chunks, 1, nbranch, mu_GP, workspace, workspace_bytes);
}

int psoap_farm_lnprob(psoap_farm* f, const double* p_dev, psoap_result* results_dev, void* stream) {
    if (!f || !p_dev || !results_dev) return fail(PSOAP_ERR_ARG, "psoap_farm_lnprob: bad arguments");
    return run_farm_graph(f, f->g, p_dev, results_dev, (cudaStream_t)stream,
                          [f](cudaStream_t s0, int pdl) { return farm_issue(f, s0, pdl); });
}

int psoap_farm_launches_per_eval(const psoap_farm* f) { return f ? f->g.launches : 0; }

int psoap_farm_destroy(psoap_farm* f) {
    delete f;
    return PSOAP_OK;
}

// ---- gradient graph of a farm -----------------------------------------------------------------------------------
size_t psoap_farm_grad_workspace_bytes(const psoap_farm* f, int nbranch) {
    if (!f || nbranch < 1) return 0;
    FarmGrad probe;
    probe.g.nbranch = std::min(nbranch, f->nitems);
    return carve_farm_grad(f, nullptr, probe);
}

int psoap_farm_grad_attach(psoap_farm* f, int nbranch, void* workspace, size_t workspace_bytes) {
    if (!f || nbranch < 1 || !workspace) return fail(PSOAP_ERR_ARG, "psoap_farm_grad_attach: bad arguments");
    if (f->grad) return fail(PSOAP_ERR_ARG, "psoap_farm_grad_attach: the farm already has a gradient graph");
    nbranch = std::min(nbranch, f->nitems);
    if (((uintptr_t)workspace & 255) || workspace_bytes < psoap_farm_grad_workspace_bytes(f, nbranch))
        return fail(PSOAP_ERR_WORKSPACE, "psoap_farm_grad_attach: workspace too small or not 256-byte aligned");
    int rc = set_kernel_attributes();
    if (rc) return rc;
    FarmGrad* q = new FarmGrad();
    q->g.nbranch = nbranch;
    carve_farm_grad(f, (char*)workspace, *q);
    std::vector<JacDesc> hj(f->nitems);
    std::vector<int64_t> Ns;
    for (const psoap_chunk& ch : f->chunks) Ns.push_back(ch.N);
    for (int it = 0; it < f->nitems; ++it) {
        const psoap_chunk& ch = f->chunks[it % f->nchunks];
        hj[it] = {ch.dates, q->item_jac[it], ch.n_epochs, (it / f->nchunks) * P_STRIDE};
    }
    cudaError_t e = cudaMemcpy(q->jdescs, hj.data(), hj.size() * sizeof(JacDesc), cudaMemcpyHostToDevice);
    rc = e != cudaSuccess ? fail(PSOAP_ERR_CUDA, std::string("farm grad descs: ") + cudaGetErrorString(e))
                          : attach_farm_graph(f, q->g, Ns, true,
                                              [f, q](cudaStream_t s0, int pdl) { return farm_grad_issue(f, *q, s0, pdl); });
    if (rc != PSOAP_OK) { delete q; return rc; }
    f->grad = q;
    return PSOAP_OK;
}

int psoap_farm_lnprob_grad(psoap_farm* f, const double* p_dev, psoap_result* results_dev, double* grad_dev,
                           void* stream) {
    if (!f || !p_dev || !results_dev || !grad_dev) return fail(PSOAP_ERR_ARG, "psoap_farm_lnprob_grad: bad arguments");
    if (!f->grad) return fail(PSOAP_ERR_ARG, "psoap_farm_lnprob_grad: no gradient graph (psoap_farm_grad_attach first)");
    FarmGrad& q = *f->grad;
    cudaStream_t st = (cudaStream_t)stream;
    int rc = run_farm_graph(f, q.g, p_dev, results_dev, st,
                            [f, &q](cudaStream_t s0, int pdl) { return farm_grad_issue(f, q, s0, pdl); });
    if (rc) return rc;
    CUDA_TRY(cudaMemcpyAsync(grad_dev, q.grad, (size_t)f->nitems * (f->norb + 2 * f->ncomp) * 8, cudaMemcpyDeviceToDevice, st));
    return PSOAP_OK;
}

// ---- prediction graph of a farm ---------------------------------------------------------------------------------
namespace {
// the checks both prediction entries make on their arguments, on the host only
bool predict_args_ok(const psoap_farm* f, int nbranch, const int64_t* m, int sigma_mode) {
    if (!f || nbranch < 1 || !m || (sigma_mode != 0 && sigma_mode != 1)) return false;
    for (int i = 0; i < f->nchunks; ++i)
        if (m[i] < 0 || m[i] > 200000 || (f->chunks[i].N < 1 && m[i] != 0)) return false;
    return true;
}
}  // namespace

size_t psoap_farm_predict_workspace_bytes(const psoap_farm* f, int nbranch, const int64_t* m, int sigma_mode) {
    if (!predict_args_ok(f, nbranch, m, sigma_mode)) return 0;
    FarmPredict probe;
    probe.g.nbranch = std::min(nbranch, f->nitems);
    return carve_farm_predict(f, m, sigma_mode, nullptr, probe);
}

int psoap_farm_predict_attach(psoap_farm* f, int nbranch, const int64_t* m, const double* const* grids, int sigma_mode,
                              void* workspace, size_t workspace_bytes, int64_t* offsets_out) {
    if (!predict_args_ok(f, nbranch, m, sigma_mode) || !grids || !workspace || !offsets_out)
        return fail(PSOAP_ERR_ARG, "psoap_farm_predict_attach: bad arguments");
    for (int i = 0; i < f->nchunks; ++i)
        for (int c = 0; c < f->ncomp; ++c)
            if (m[i] > 0 && !grids[(size_t)i * f->ncomp + c])
                return fail(PSOAP_ERR_ARG, "psoap_farm_predict_attach: null grid of chunk " + std::to_string(i));
    if (f->pred) return fail(PSOAP_ERR_ARG, "psoap_farm_predict_attach: the farm already has a prediction graph");
    nbranch = std::min(nbranch, f->nitems);
    if (((uintptr_t)workspace & 255) || workspace_bytes < psoap_farm_predict_workspace_bytes(f, nbranch, m, sigma_mode))
        return fail(PSOAP_ERR_WORKSPACE, "psoap_farm_predict_attach: workspace too small or not 256-byte aligned");
    int rc = set_kernel_attributes();
    if (rc) return rc;
    const int nitems = f->nitems, nchunks = f->nchunks;
    FarmPredict* q = new FarmPredict();
    q->g.nbranch = nbranch;
    q->sigma_mode = sigma_mode;
    q->m.assign(m, m + nchunks);
    q->grids.assign(grids, grids + (size_t)nchunks * f->ncomp);
    carve_farm_predict(f, m, sigma_mode, (char*)workspace, *q);
    // the LPT weight of an item is its bordered dimension Nt (cubed by lpt_items); items of chunks with m = 0 take no work
    std::vector<int64_t> cost(nchunks);
    for (int i = 0; i < nchunks; ++i) cost[i] = m[i] > 0 ? predict_item_dims(f->ncomp, f->chunks[i].N, m[i]).Nt : 0;
    // the records of items with m = 0 are never written by the graph: they read 0 (lnlike, logdet, quad, info)
    cudaError_t e = cudaMemset(q->g.results, 0, (size_t)nitems * 4 * 8);
    rc = e != cudaSuccess ? fail(PSOAP_ERR_CUDA, std::string("farm predict results: ") + cudaGetErrorString(e))
                          : attach_farm_graph(f, q->g, cost, true, [f, q](cudaStream_t s0, int pdl) {
                                return farm_predict_issue(f, *q, s0, pdl, q->cap_delta, q->cap_sigma);
                            });
    if (rc != PSOAP_OK) { delete q; return rc; }
    f->pred = q;
    std::copy(q->delta_off.begin(), q->delta_off.end(), offsets_out);
    std::copy(q->sigma_off.begin(), q->sigma_off.end(), offsets_out + nitems + 1);
    return PSOAP_OK;
}

int psoap_farm_predict(psoap_farm* f, const double* p_dev, double* delta_dev, double* sigma_dev,
                       psoap_result* results_dev, void* stream) {
    if (!f || !p_dev || !delta_dev || !sigma_dev || !results_dev)
        return fail(PSOAP_ERR_ARG, "psoap_farm_predict: bad arguments");
    if (!f->pred) return fail(PSOAP_ERR_ARG, "psoap_farm_predict: no prediction graph (psoap_farm_predict_attach first)");
    FarmPredict& q = *f->pred;
    cudaStream_t st = (cudaStream_t)stream;
    // direct issue writes into the caller's buffers; the captured graph into its own, copied out after the replay
    int rc = run_farm_graph(f, q.g, p_dev, results_dev, st, [f, &q, delta_dev, sigma_dev](cudaStream_t s0, int pdl) {
        return farm_predict_issue(f, q, s0, pdl, delta_dev, sigma_dev);
    });
    if (rc) return rc;
    if (!q.g.direct) {
        CUDA_TRY(cudaMemcpyAsync(delta_dev, q.cap_delta, (size_t)q.delta_off[f->nitems] * 8, cudaMemcpyDeviceToDevice, st));
        CUDA_TRY(cudaMemcpyAsync(sigma_dev, q.cap_sigma, (size_t)q.sigma_off[f->nitems] * 8, cudaMemcpyDeviceToDevice, st));
    }
    return PSOAP_OK;
}

// Times the trailing-update kernel (syrk3_kernel, the dominant kernel of the path) alone: `reps` launches of the rank-K update (K a multiple of 128) of an m x m lower triangle (m a multiple of 128), CUDA events on a private
// stream.  flops_per_launch is the algorithmic count K * m * (m + 1) (DSYRK convention).
int psoap_bench_syrk(int64_t m, int K, int reps, double* avg_ms_out, double* flops_per_launch_out) {
    return psoap_bench_syrk_split(m, K, reps, g_tail_split, avg_ms_out, flops_per_launch_out);
}

// The same with the quarter-tile tail (syrk_split) forced on or off: the configuration that ships is
// psoap_bench_syrk's; this entry exists so that the bench line can show what the tail costs the kernel when it runs alone.
int psoap_bench_syrk_split(int64_t m, int K, int reps, int tail_split, double* avg_ms_out, double* flops_per_launch_out) {
    if (m < NB || m % NB || reps < 1 || !avg_ms_out || K < NB || K % NB || K > 2048)
        return fail(PSOAP_ERR_ARG, "psoap_bench_syrk: bad arguments");
    int rc = set_kernel_attributes();
    if (rc) return rc;
    double *W = nullptr, *P = nullptr, *y = nullptr, *r = nullptr;
    CUDA_TRY(cudaMalloc(&W, (size_t)m * m * 8));
    CUDA_TRY(cudaMalloc(&P, (size_t)m * K * 8));
    CUDA_TRY(cudaMalloc(&y, NB * 8));
    CUDA_TRY(cudaMalloc(&r, (size_t)m * 8));
    CUDA_TRY(cudaMemset(W, 0, (size_t)m * m * 8));
    CUDA_TRY(cudaMemset(y, 0, NB * 8));
    CUDA_TRY(cudaMemset(r, 0, (size_t)m * 8));
    std::vector<double> hp((size_t)m * K);
    for (size_t i = 0; i < hp.size(); ++i) hp[i] = 1e-3 * (double)((i * 2654435761u) % 1000) - 0.5;
    CUDA_TRY(cudaMemcpy(P, hp.data(), hp.size() * 8, cudaMemcpyHostToDevice));
    cudaStream_t st;
    CUDA_TRY(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
    cudaEvent_t e0, e1;
    CUDA_TRY(cudaEventCreate(&e0));
    CUDA_TRY(cudaEventCreate(&e1));
    const int R = (int)(m / NB), ntiles = R * (R + 1);
    SyrkSrc src;
    src.W = W; src.ld = m; src.row0 = 0; src.res_row0 = 0; src.kbeg = 0; src.kend = K; src.P = P; src.ldp = m; src.part = 0; src.ncol1 = 2;
    const SyrkSplit sp = syrk_split(ntiles, false, tail_split != 0);
    CUtensorMap mapPa, mapPb, mapQa, mapQb;
    rc = make_tensor_map(&mapPa, P, (uint64_t)m, (uint64_t)K, (uint64_t)m, SA);
    if (!rc) rc = make_tensor_map(&mapPb, P, (uint64_t)m, (uint64_t)K, (uint64_t)m, SB);
    if (!rc) rc = make_tensor_map(&mapQa, P, (uint64_t)m, (uint64_t)K, (uint64_t)m, Shape<2>::SA);
    if (!rc) rc = make_tensor_map(&mapQb, P, (uint64_t)m, (uint64_t)K, (uint64_t)m, Shape<2>::SB);
    if (rc) return rc;
    auto launch = [&]() {
        syrk3_kernel<1><<<R + sp.nctas + sp.nquarters, 256, SYRK1_SMEM, st>>>(src, sp.nmain, sp.nctas, R, y, r, 0, mapPa, mapPb,
                                                                              mapQa, mapQb);
        ++g_launches;
    };
    for (int w = 0; w < 2; ++w) launch();
    cudaEventRecord(e0, st);
    for (int i = 0; i < reps; ++i) launch();
    cudaEventRecord(e1, st);
    CUDA_TRY(cudaEventSynchronize(e1));
    float ms = 0;
    cudaEventElapsedTime(&ms, e0, e1);
    cudaEventDestroy(e0); cudaEventDestroy(e1); cudaStreamDestroy(st);
    cudaFree(W); cudaFree(P); cudaFree(y); cudaFree(r);
    *avg_ms_out = ms / reps;
    // algorithmic flops of the rank-K update of a lower triangle (the DSYRK convention k n (n+1)); the kernel also
    // computes the upper halves of the diagonal tiles, K m 127 flops that are not counted
    if (flops_per_launch_out) *flops_per_launch_out = (double)K * (double)m * (double)(m + 1);
    return PSOAP_OK;
}

// The INTERNAL fill of the likelihood (fill_lower_kernel: lower triangle of K + sigma^2 I, front padding, fused
// Doppler shift) written into a caller-provided column-major matrix, for the entry-wise parity tests against
// matrix_functions.pyx:125-144 and for timing.  epoch/vel null: lwl_f/g/h are the already shifted per-component
// vectors; otherwise lwl_f is the base vector and vel [ncomp, n_epochs] the velocity table (data.py:40-63).
int psoap_debug_fill_lower(int ncomp, int64_t N, const double* lwl_f, const double* lwl_g, const double* lwl_h,
                           const int32_t* epoch, const double* vel, int n_epochs, const double* fl, const double* sigma,
                           const double* amp, const double* l, double mu_GP, double* W, int64_t ld, double* rvec,
                           void* stream) {
    if (ncomp < 1 || ncomp > 3 || N < 1 || !lwl_f || !fl || !sigma || !amp || !l || !W || !rvec)
        return fail(PSOAP_ERR_ARG, "psoap_debug_fill_lower: bad arguments");
    const int64_t Np = padded_dim(N);
    if (ld < Np || (ld & 1) || ((uintptr_t)W & 15)) return fail(PSOAP_ERR_ARG, "psoap_debug_fill_lower: ld/alignment");
    GpParams gp;
    make_gp(ncomp, amp, l, &gp);
    ZSource zs = direct_z(lwl_f, lwl_g, lwl_h);
    if (epoch && vel) { zs.epoch = epoch; zs.vel = vel; zs.n_epochs = n_epochs; zs.shift = 1; }
    double* scratch = nullptr;   // accumulators + info word the kernel resets
    CUDA_TRY(cudaMalloc(&scratch, 256));
    FactorWs ws{};
    ws.rvec = rvec; ws.acc = scratch; ws.info = (int*)(scratch + 16); ws.Nt = Np;
    int rc = launch_fill_lower(ncomp, (cudaStream_t)stream, W, ld, (int)(Np / NB), (int)(Np - N), zs, sigma, fl, mu_GP, gp, ws);
    cudaError_t e = cudaStreamSynchronize((cudaStream_t)stream);
    cudaFree(scratch);
    if (rc) return rc;
    if (e != cudaSuccess) return fail(PSOAP_ERR_CUDA, std::string("psoap_debug_fill_lower: ") + cudaGetErrorString(e));
    return PSOAP_OK;
}

// Times a fill kernel alone on the caller's (already Doppler-shifted, device) ln-wavelength vectors:
// kind 0 = fill_lower_kernel (the likelihood's internal fill, column-major lower triangle, 4 N^2 algorithmic bytes),
// kind 1 = fill_full_kernel (operator surface fill_V11_*, row-major both triangles, 8 N^2 bytes).  `reps` launches
// between CUDA events on a private stream; the matrix is allocated here.
int psoap_bench_fill(int kind, int ncomp, int64_t N, const double* lwl_f, const double* lwl_g, const double* lwl_h,
                     const double* amp, const double* l, int reps, double* avg_ms_out) {
    if (kind < 0 || kind > 1 || ncomp < 1 || ncomp > 3 || N < 1 || !lwl_f || !amp || !l || reps < 1 || !avg_ms_out)
        return fail(PSOAP_ERR_ARG, "psoap_bench_fill: bad arguments");
    const int64_t Np = padded_dim(N);
    double *W = nullptr, *vec = nullptr;
    CUDA_TRY(cudaMalloc(&W, (size_t)Np * Np * 8));
    CUDA_TRY(cudaMalloc(&vec, (size_t)(3 * Np + 64) * 8));
    CUDA_TRY(cudaMemset(vec, 0, (size_t)(3 * Np + 64) * 8));
    cudaStream_t st;
    CUDA_TRY(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
    cudaEvent_t e0, e1;
    CUDA_TRY(cudaEventCreate(&e0));
    CUDA_TRY(cudaEventCreate(&e1));
    GpParams gp;
    make_gp(ncomp, amp, l, &gp);
    ZSource zs = direct_z(lwl_f, lwl_g, lwl_h);
    FactorWs ws{};
    ws.rvec = vec; ws.acc = vec + 3 * Np; ws.info = (int*)(vec + 3 * Np + 16); ws.Nt = Np;
    const double* sigma = vec + Np;   // zeros
    const double* fl = vec + 2 * Np;  // zeros
    int rc = PSOAP_OK;
    auto launch = [&]() {
        if (kind == 0) rc = launch_fill_lower(ncomp, st, W, Np, (int)(Np / NB), (int)(Np - N), zs, sigma, fl, 1.0, gp, ws);
        else rc = psoap_fill_v11(ncomp, W, N, N, lwl_f, lwl_g, lwl_h, amp, l, st);
    };
    for (int w = 0; w < 2 && !rc; ++w) launch();
    cudaEventRecord(e0, st);
    for (int i = 0; i < reps && !rc; ++i) launch();
    cudaEventRecord(e1, st);
    cudaError_t e = cudaEventSynchronize(e1);
    float ms = 0;
    cudaEventElapsedTime(&ms, e0, e1);
    cudaEventDestroy(e0); cudaEventDestroy(e1); cudaStreamDestroy(st);
    cudaFree(W); cudaFree(vec);
    if (rc) return rc;
    if (e != cudaSuccess) return fail(PSOAP_ERR_CUDA, std::string("psoap_bench_fill: ") + cudaGetErrorString(e));
    *avg_ms_out = ms / reps;
    return PSOAP_OK;
}

// Host-side replay of the trailing-update tile enumeration (no device work): writes (row, column-tile) of every
// tile of a launch over R row tiles; returns the tile count, or -1 when `cap` is too small.
int psoap_debug_syrk_tiles(int R, int part, int ncol1, int* rows_out, int* cols_out, int cap) {
    SyrkSrc src{};
    src.part = part; src.ncol1 = ncol1;
    const int n = syrk_ntiles(R, part, ncol1);
    if (n > cap) return -1;
    for (int t = 0; t < n; ++t) src.decode(t, rows_out[t], cols_out[t]);
    return n;
}

#ifdef PSOAP_TIMELINE
// Lab builds only (tools/timeline.py): copies the CTA time stamps out (7 int64 per record) and resets the counter.
extern "C" int psoap_debug_timeline(long long* out, int cap) {
    unsigned n = 0;
    CUDA_TRY(cudaDeviceSynchronize());
    CUDA_TRY(cudaMemcpyFromSymbol(&n, g_tl_n, sizeof(n)));
    n = std::min(n, TL_CAP);
    std::vector<TlRec> h(n);
    if (n) CUDA_TRY(cudaMemcpyFromSymbol(h.data(), g_tl, (size_t)n * sizeof(TlRec)));
    const int m = std::min<int>((int)n, cap);
    for (int i = 0; i < m; ++i) {
        out[7 * i] = (long long)h[i].t_in; out[7 * i + 1] = (long long)h[i].t_go; out[7 * i + 2] = (long long)h[i].t_out;
        out[7 * i + 3] = h[i].kernel; out[7 * i + 4] = h[i].block; out[7 * i + 5] = h[i].nblocks; out[7 * i + 6] = h[i].smid;
    }
    const unsigned zero = 0;
    CUDA_TRY(cudaMemcpyToSymbol(g_tl_n, &zero, sizeof(zero)));
    return (int)n;
}
#endif

int psoap_fp64_peak_tflops(double* tflops_out) {
    if (!tflops_out) return fail(PSOAP_ERR_ARG, "psoap_fp64_peak_tflops: null");
    int dev = 0, sms = 0;
    CUDA_TRY(cudaGetDevice(&dev));
    CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    double* out = nullptr;
    CUDA_TRY(cudaMalloc(&out, (size_t)sms * 512 * 8));
    cudaEvent_t e0, e1;
    CUDA_TRY(cudaEventCreate(&e0));
    CUDA_TRY(cudaEventCreate(&e1));
    const int iters = 20000;
    float best = 1e30f;
    for (int r = 0; r < 4; ++r) {
        cudaEventRecord(e0);
        dmma_peak_kernel<<<sms, 512>>>(out, iters);
        cudaEventRecord(e1);
        CUDA_TRY(cudaEventSynchronize(e1));
        float ms = 0;
        cudaEventElapsedTime(&ms, e0, e1);
        if (r > 0 && ms < best) best = ms;
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1); cudaFree(out);
    *tflops_out = 2.0 * 256 * 8 * (double)iters * 16 * sms / (best * 1e-3) * 1e-12;
    return PSOAP_OK;
}

}  // extern "C"
