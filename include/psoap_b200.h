/*
 * psoap_b200.h — C ABI of the B200-native (sm_100a) PSOAP GP log-likelihood path.
 *
 * Drop-in boundary for the reference's only native/third-party interfaces on this path:
 *   psoap/matrix_functions.pyx (Cython fills)              -> psoap_fill_v11 / psoap_fill_v12
 *   scipy.linalg.cho_factor / cho_solve (LAPACK dpotrf/s)  -> fused inside psoap_lnlike / psoap_schur
 *   psoap/data.py lredshift / replicate_wls                -> psoap_replicate_wls (and fused in the farm fill)
 *   psoap/orbit.py get_velocities                          -> psoap_orbit_velocities
 *   psoap/sample_parallel.py Worker.lnprob + master lnprob -> psoap_farm_*
 * Paths are relative to the reference repository root.  All arithmetic is IEEE FP64.
 *
 * Conventions
 *   - plain C types only; every `*_dev` / "device" pointer is a CUDA device pointer on the current device;
 *     `stream` is a cudaStream_t passed as void* (NULL = default stream); calls are asynchronous on that
 *     stream unless stated otherwise.
 *   - return value: 0 = ok; <0 = argument/CUDA error (message via psoap_last_error()).  Numerical failure
 *     (non-positive pivot, LAPACK "info > 0") is NOT an error return: it is reported in the result record,
 *     because the reference turns it into the value -inf (psoap/covariance.py:326-327).
 *   - there is no CPU fallback: without a CUDA device every compute entry point returns PSOAP_ERR_CUDA.
 */
#ifndef PSOAP_B200_H
#define PSOAP_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PSOAP_OK 0
#define PSOAP_ERR_ARG (-1)
#define PSOAP_ERR_CUDA (-2)
#define PSOAP_ERR_WORKSPACE (-3)

/* orbital models, psoap/orbit.py:490 `models` */
#define PSOAP_SB1 1
#define PSOAP_SB2 2
#define PSOAP_ST1 3
#define PSOAP_ST2 4
#define PSOAP_ST3 5

/* Result record written (on the device) by psoap_lnlike and, per chunk, by the farm. */
typedef struct {
    double lnlike; /* -0.5 (quad + logdet), or -inf when info != 0 / a sentinel fired (covariance.py:331) */
    double logdet; /* sum_i 2 log L_ii                                   (covariance.py:329)            */
    double quad;   /* (fl - mu)^T K^-1 (fl - mu)                                                       */
    double info;   /* 0, or 1-based index of the first non-positive pivot (LAPACK dpotrf info), as a double */
} psoap_result;

/* One spectral chunk resident on the device (what sample_parallel.Worker keeps after INIT, :126-166). */
typedef struct {
    int64_t N;            /* number of unmasked pixels                                                   */
    int32_t n_epochs;
    int32_t reserved;     /* 0, or on the FIRST chunk: low byte 3 | 7 forces the chain-link kernels of the whole farm, the next
                           * byte 2 | 4 | 8 its panels per trailing update (a farm partitioned over ranks passes the same
                           * value everywhere: bits independent of the GPU count) */
    const double *lwl;    /* [N] ln-wavelength of the masked, epoch-major flattened pixels (data.py:126)  */
    const int32_t *epoch; /* [N] epoch index of every pixel (what the mask broadcast in data.py:61 encodes) */
    const double *fl;     /* [N] flux                                                                    */
    const double *sigma;  /* [N] noise (already multiplied by `soften`, sample_parallel.py:141)           */
    const double *dates;  /* [n_epochs] observation dates (date1D)                                       */
} psoap_chunk;

const char *psoap_last_error(void);
int psoap_version(void);
int psoap_device_count(void);

/* ---- fills: psoap/matrix_functions.pyx --------------------------------------------------------------- */
/* fill_V11_f (:21-57, ncomp=1), fill_V11_f_g (:101-144, ncomp=2), fill_V11_f_g_h (:151-201, ncomp=3).
 * mat: device, row-major [N, ld] (ld >= N, in elements), both triangles and the diagonal are written.
 * lwl_g / lwl_h may be NULL when unused.  amp, l: HOST arrays of ncomp doubles. */
int psoap_fill_v11(int ncomp, double *mat_dev, int64_t ld, int64_t N, const double *lwl_f_dev,
                   const double *lwl_g_dev, const double *lwl_h_dev, const double *amp, const double *l,
                   void *stream);
/* Same for HOST arrays (mat and the ln-wavelength vectors in host memory; synchronous, the N x N result crosses PCIe):
 * the entry a seam at matrix_functions.pyx binds, `fill_V11_f(mat, lwl_f, amp_f, l_f)` ->
 * `psoap_fill_v11_host(1, &mat[0,0], mat.shape[1], N, &lwl_f[0], NULL, NULL, &amp_f, &l_f)`. */
int psoap_fill_v11_host(int ncomp, double *mat, int64_t ld, int64_t N, const double *lwl_f, const double *lwl_g,
                        const double *lwl_h, const double *amp, const double *l);
/* fill_V12_f (:63-94): mat row-major [M, ld]; M = len(lwl_rows), N = len(lwl_cols);
 * mat[i,j] = amp^2 exp(-0.5 c^2 (lwl_cols[j] - lwl_rows[i])^2 / l^2). */
int psoap_fill_v12(double *mat_dev, int64_t ld, int64_t M, int64_t N, const double *lwl_rows_dev,
                   const double *lwl_cols_dev, double amp, double l, void *stream);

/* Sum over ncomp components of fill_V12_f (V12_f + V12_g (+ V12_h), psoap/covariance.py:167-171,:272-278).
 * rows, cols: HOST arrays of ncomp device pointers; amp, l: HOST arrays of ncomp doubles. */
int psoap_fill_v12n(int ncomp, double *mat_dev, int64_t ld, int64_t M, int64_t N, const double *const *rows_dev,
                    const double *const *cols_dev, const double *amp, const double *l, void *stream);

/* ---- Doppler shift: psoap/data.py:25-63 -------------------------------------------------------------- */
/* out[c*N + k] = lwl[k] + (-vel[c*n_epochs + epoch[k]]) / c_kms */
int psoap_replicate_wls(double *out_dev, const double *lwl_dev, const int32_t *epoch_dev, int64_t N,
                        const double *vel_dev, int ncomp, int n_epochs, void *stream);

/* ---- orbits: psoap/orbit.py get_velocities (:94-115, :148-170, :295-320, :390-417, :463-487) --------- */
/* p_orb_dev: orbital parameters in utils.registered_params order (utils.py:4-8) on the device.
 * vel_dev: [ncomp, n_epochs].  flag_dev (may be NULL): set to 1 if any |v| >= c_kms (sample_parallel.py:186). */
int psoap_orbit_velocities(int model, const double *p_orb_dev, const double *dates_dev, int n_epochs,
                           double *vel_dev, int *flag_dev, void *stream);
int psoap_model_ncomp(int model);
int psoap_model_norb(int model);

/* ---- likelihood: psoap/covariance.py:299-376 --------------------------------------------------------- */
size_t psoap_lnlike_workspace_bytes(int64_t N);
/* lnlike_f / lnlike_f_g / lnlike_f_g_h by ncomp.  All vectors are device pointers of length N; amp, l are
 * HOST arrays of ncomp doubles.  workspace_dev: >= psoap_lnlike_workspace_bytes(N) bytes, 256-byte aligned.
 * Negative amp or l gives lnlike = -inf without touching the device matrix (covariance.py:317,:339,:362).
 * N = 0 (an empty chunk, vectors may be null) gives -0.0 like the reference, whose sums then run over nothing. */
int psoap_lnlike(int ncomp, int64_t N, const double *lwl_f_dev, const double *lwl_g_dev, const double *lwl_h_dev,
                 const double *fl_dev, const double *sigma_dev, const double *amp, const double *l, double mu_GP,
                 void *workspace_dev, size_t workspace_bytes, psoap_result *result_dev, void *stream);
/* Same with HOST vectors: uploads, evaluates and downloads synchronously on an internal stream, with an
 * internally cached device workspace.  This is the entry a C/ctypes caller with host arrays binds. */
int psoap_lnlike_host(int ncomp, int64_t N, const double *lwl_f, const double *lwl_g, const double *lwl_h,
                      const double *fl, const double *sigma, const double *amp, const double *l, double mu_GP,
                      psoap_result *result);
/* The envelope the last psoap_lnlike call on this workspace computed on the device: *tend_dev points at int[T + 1]
 * (T = padded(N) / 128 row blocks); tend[e], e >= 1, is the first row block from which every row of K is exactly zero
 * in block columns [0, e).  The factorisation's launches for panels before e stop there. */
int psoap_lnlike_envelope_view(void *workspace_dev, int64_t N, int **tend_dev, int *T);

/* ---- prediction: psoap/covariance.py:81-297 (Schur complement of a bordered matrix) ------------------- */
/* In place on a column-major device matrix S [n + m, ld]: the leading n x n block (lower triangle) is
 * K + sigma^2 I, rows n.. hold the border [C | A] (lower triangle of A).  On return the trailing m x m
 * block (lower triangle) holds A - C K^-1 C^T; result->logdet/info describe the leading block.
 * workspace_dev: >= psoap_schur_workspace_bytes(n, m). */
size_t psoap_schur_workspace_bytes(int64_t n, int64_t m);
int psoap_schur(double *S_dev, int64_t ld, int64_t n, int64_t m, void *workspace_dev, size_t workspace_bytes,
                psoap_result *result_dev, void *stream);
/* Views into a Schur workspace: the residual vector r [padded(n) + padded(m)] (set it before psoap_schur:
 * fl - mu on the data rows, 0 elsewhere; afterwards rows >= padded(n) hold -C K^-1 (fl - mu)), the
 * accumulators (zero them before the call) and the pivot info word (zero it before the call). */
int psoap_schur_views(void *workspace_dev, int64_t n, int64_t m, double **rvec_dev, double **acc_dev,
                      int **info_dev);

/* The whole prediction as ONE call (psoap/covariance.py: predict_f :25-54, predict_f_g :81-148, predict_f_g_sum :151-187,
 * predict_f_g_h :190-251, predict_f_g_h_sum :253-297): builds the bordered matrix on the device (lower triangle only,
 * no N^2 memset), eliminates the data block with the likelihood's kernels and reads the Schur complement out.
 *   mode 0: components stacked, M = ncomp * m outputs: A = blockdiag(K_c(predict_c)), C = [K_c(predict_c, data_c)]_c
 *   mode 1: summed process, M = m:                     A = sum_c K_c(predict_c) + nugget I, C = sum_c K_c(predict_c, data_c)
 *   mode 2: as 1 with the cross block transposed (the mean of predict_f_g_h_sum multiplies by V12.T, :294); needs m == n
 * lwl_data / lwl_predict: HOST arrays of ncomp device pointers ([n] / [m] each); amp, l: HOST arrays of ncomp doubles.
 * delta_out_dev [M]      = C K^-1 (fl - resid_mu)   (the caller adds its mean: mu_f/mu_g..., the reference's hard-coded
 *                          `fl - 1.0` of :140,:184,:248 is resid_mu = 1.0)
 * Sigma_out_dev [M, M]   = A - C K^-1 C^T, row-major, both triangles; may be NULL (get_Sigma=False)
 * result_dev             logdet / info of the data block: info != 0 is the reference's LinAlgError (:113 has no try).
 * workspace_dev: >= psoap_predict_workspace_bytes(...) bytes, 256-byte aligned.  Asynchronous on `stream`. */
size_t psoap_predict_workspace_bytes(int ncomp, int mode, int64_t n, int64_t m);
int psoap_predict(int ncomp, int mode, int64_t n, int64_t m, const double *const *lwl_data_dev, const double *fl_dev,
                  const double *sigma_dev, const double *const *lwl_predict_dev, const double *amp, const double *l,
                  double resid_mu, double nugget, double *delta_out_dev, double *Sigma_out_dev, void *workspace_dev,
                  size_t workspace_bytes, psoap_result *result_dev, void *stream);
/* Same with HOST vectors in and HOST delta / Sigma / result out (synchronous; device memory is allocated and freed
 * inside): the entry a C caller without device buffers binds. */
int psoap_predict_host(int ncomp, int mode, int64_t n, int64_t m, const double *const *lwl_data, const double *fl,
                       const double *sigma, const double *const *lwl_predict, const double *amp, const double *l,
                       double resid_mu, double nugget, double *delta_out, double *Sigma_out, psoap_result *result);

/* ---- gradient of the log-likelihood ------------------------------------------------------------------- */
/* lnlike_f / _f_g / _f_g_h (as psoap_lnlike) together with its exact gradient:
 *   grad_hyp_dev [2 ncomp + 1]    d lnlike / d(amp_f, l_f, amp_g, l_g, amp_h, l_h (first 2 ncomp), mu_GP)
 *   grad_lwl_dev [ncomp, N]       d lnlike / d lwl_c[i] (the shifted ln-wavelengths), or NULL when not wanted.
 * K^-1 comes from eliminating the data block of [[K, I], [I, 0]] with the likelihood's kernels (about three times the
 * work of psoap_lnlike for large N); every sum runs in a fixed order, so the result is bit-identical from run to run.
 * Arguments, the negative-hyper-parameter and N = 0 conventions and the stream use are those of psoap_lnlike; when
 * lnlike is -inf (negative hyper-parameters, info != 0) every gradient entry is NaN; N = 0 gives -0.0 and zeros.
 * workspace_dev: >= psoap_lnlike_grad_workspace_bytes(ncomp, N) bytes, 256-byte aligned. */
size_t psoap_lnlike_grad_workspace_bytes(int ncomp, int64_t N);
int psoap_lnlike_grad(int ncomp, int64_t N, const double *lwl_f_dev, const double *lwl_g_dev, const double *lwl_h_dev,
                      const double *fl_dev, const double *sigma_dev, const double *amp, const double *l, double mu_GP,
                      void *workspace_dev, size_t workspace_bytes, psoap_result *result_dev, double *grad_hyp_dev,
                      double *grad_lwl_dev, void *stream);
/* Views into a gradient workspace after psoap_lnlike_grad (their offsets depend on N alone): -K^-1 as the lower
 * triangle of a column-major [N, N] block with leading dimension *ld (data order), and -alpha = -K^-1 (fl - mu) [N]. */
int psoap_lnlike_grad_views(void *workspace_dev, int64_t N, double **neg_kinv_dev, int64_t *ld, double **neg_alpha_dev);
/* One chunk of the farm with its gradient for the full registered parameter vector p_dev (orbital then GP,
 * utils.py:4-8; on the device): orbit velocities and sentinel, the Doppler-shifted fill, the identity-bordered
 * elimination, the contraction, the per-epoch sum and the orbit Jacobian.  grad_p_dev [norb + 2 ncomp]; NaN when
 * lnlike is -inf (|v| >= c, a negative GP hyper-parameter, info != 0).  chunk->reserved is ignored (the direct API's
 * launch choices apply).  workspace_dev: >= psoap_chunk_lnprob_grad_workspace_bytes(model, N, n_epochs) bytes. */
size_t psoap_chunk_lnprob_grad_workspace_bytes(int model, int64_t N, int32_t n_epochs);
int psoap_chunk_lnprob_grad(int model, const psoap_chunk *chunk, const double *p_dev, double mu_GP, void *workspace_dev,
                            size_t workspace_bytes, psoap_result *result_dev, double *grad_p_dev, void *stream);
/* d v_c[ep] / d p_k of psoap_orbit_velocities: jac_dev [ncomp][n_epochs][norb], p_orb_dev in registered order. */
int psoap_orbit_jacobian(int model, const double *p_orb_dev, const double *dates_dev, int n_epochs, double *jac_dev,
                         void *stream);

/* ---- expected Fisher information of one chunk ---------------------------------------------------------- */
/* psoap_chunk_lnprob_grad plus fisher_dev [n_params][n_params] (row-major, symmetric bit for bit, n_params =
 * norb + 2 ncomp):  F_ab = 1/2 tr(K^-1 dK/dp_a K^-1 dK/dp_b) in the full registered parameter vector.  NaN everywhere
 * when lnlike is -inf.  The gamma row and column are exactly zero (the covariance depends on velocity differences
 * only).  result_dev and grad_p_dev receive exactly what psoap_chunk_lnprob_grad writes; grad_p_dev may be NULL.
 * Bit-reproducible: no floating-point atomics.  workspace_dev: >= psoap_chunk_fisher_workspace_bytes(model, N,
 * n_epochs) bytes, 256-byte aligned: the gradient's identity-bordered matrix plus one N x N product per parameter,
 * about (4 + n_params) 8 N^2 bytes. */
size_t psoap_chunk_fisher_workspace_bytes(int model, int64_t N, int32_t n_epochs);
int psoap_chunk_fisher(int model, const psoap_chunk *chunk, const double *p_dev, double mu_GP, void *workspace_dev,
                       size_t workspace_bytes, psoap_result *result_dev, double *grad_p_dev, double *fisher_dev,
                       void *stream);
/* Views into a Fisher workspace after psoap_chunk_fisher: *Tb = padded N / 128, the tile flags [Tb][Tb] (1 where an
 * exponential factor of the covariance is non-zero in the 128 x 128 tile) and the k range [Tb][2] (first and last
 * flagged row block of each block column) that the products run over. */
int psoap_chunk_fisher_views(void *workspace_dev, int model, int64_t N, int32_t n_epochs, uint8_t **flags_dev,
                             int **krange_dev, int *Tb);

/* ---- chunk farm: psoap/sample_parallel.py:168-198, :371-390 ------------------------------------------ */
typedef struct psoap_farm psoap_farm;
size_t psoap_farm_workspace_bytes(int nchunks, const int64_t *N, const int32_t *n_epochs, int nbranch);
/* chunks: HOST array of descriptors whose pointers are device pointers that stay valid for the farm's life.
 * nbranch: number of chunks evaluated concurrently (independent CUDA-graph branches). */
int psoap_farm_create(psoap_farm **farm, int model, int nchunks, const psoap_chunk *chunks, int nbranch,
                      double mu_GP, void *workspace_dev, size_t workspace_bytes);
/* p_dev: full registered parameter vector (orbital then GP, utils.py:4-8) on the device.
 * results_dev: [nchunks] records; lnlike is -inf for |v| >= c (sample_parallel.py:186-187), negative
 * hyper-parameters, or a non-positive pivot. */
int psoap_farm_lnprob(psoap_farm *farm, const double *p_dev, psoap_result *results_dev, void *stream);
/* Batched variant (ensemble samplers, SURVEY.md §8f-2): nprop proposals are evaluated by one graph launch; every
 * (proposal, chunk) pair is an independent work item.  p_dev of psoap_farm_lnprob is then [nprop][n_params]
 * contiguous and results_dev is [nprop][nchunks]. */
size_t psoap_farm_workspace_bytes_batched(int nchunks, const int64_t *N, const int32_t *n_epochs, int nprop,
                                          int nbranch);
int psoap_farm_create_batched(psoap_farm **farm, int model, int nchunks, const psoap_chunk *chunks, int nprop,
                              int nbranch, double mu_GP, void *workspace_dev, size_t workspace_bytes);
int psoap_farm_launches_per_eval(const psoap_farm *farm);
/* Frees the farm's streams, events and graph, and its gradient and prediction graphs when attached (not the workspaces). */
int psoap_farm_destroy(psoap_farm *farm);

/* Gradient graph of a farm: every (proposal, chunk) pair through the steps of psoap_chunk_lnprob_grad, nbranch pairs in
 * flight, captured into a second CUDA graph beside the likelihood's (which, with its workspace and launch count, is left
 * as it is).  A farm that never attaches one allocates and captures nothing for it.
 * psoap_farm_grad_workspace_bytes: bytes the attach needs for nbranch branches (each holds the identity-bordered
 * matrix of the largest chunk, 8 (2 padded(N))^2 bytes, plus its group buffers), 0 for a null farm or nbranch < 1.
 * psoap_farm_grad_attach: captures the graph (once per farm); workspace_dev >= psoap_farm_grad_workspace_bytes(farm,
 * nbranch) bytes, 256-byte aligned, valid for the farm's life.  Launch choices follow psoap_chunk.reserved as the
 * likelihood graph's do; look-ahead is taken where the reserved chain is 7, so that with the reserved value set the
 * gradient's bits depend neither on nbranch nor on how the chunks are partitioned over ranks. */
size_t psoap_farm_grad_workspace_bytes(const psoap_farm *farm, int nbranch);
int psoap_farm_grad_attach(psoap_farm *farm, int nbranch, void *workspace_dev, size_t workspace_bytes);
/* p_dev: [nprop][n_params] contiguous, as psoap_farm_lnprob.  results_dev: [nprop][nchunks] records.
 * grad_dev: [nprop][nchunks][n_params], the gradient of each pair's lnlike for the full registered vector (orbital then
 * GP); a row is NaN where that pair's lnlike is -inf (|v| >= c, a negative GP value, info != 0), other rows are
 * unaffected.  PSOAP_ERR_ARG before psoap_farm_grad_attach.  Every sum runs in a fixed order: the rows are
 * bit-identical from call to call. */
int psoap_farm_lnprob_grad(psoap_farm *farm, const double *p_dev, psoap_result *results_dev, double *grad_dev,
                           void *stream);

/* Prediction graph of a farm: the component spectra of every chunk at every proposal, psoap_predict mode 0
 * (psoap/covariance.py:81-148 predict_f_g, :190-251 predict_f_g_h, as scripts/psoap_retrieve_SB2.py / _ST3.py call them)
 * on the farm's resident pixels shifted by each proposal's velocities, nbranch (proposal, chunk) items in flight,
 * captured into a third CUDA graph beside the likelihood's and the gradient's (both left as they are).  A farm that
 * never attaches one allocates and captures nothing for it.
 * m: [nchunks] grid points per component of each chunk (0: the chunk takes no work; a chunk without pixels must have 0).
 * grids: [nchunks][ncomp] DEVICE pointers to each chunk's rest-frame ln-wavelength grid of each component, m[i] values
 * each; captured into the graph, so they stay valid for the farm's life.  sigma_mode 0 writes Sigma, 1 only its diagonal.
 * psoap_farm_predict_workspace_bytes: bytes the attach needs, 0 for bad arguments.  Each branch holds the bordered matrix
 * of the largest item, 8 (padded(N) + padded(ncomp m))^2 bytes, plus its factorisation scratch; the graph's outputs are
 * held as well.
 * psoap_farm_predict_attach: captures the graph (once per farm).  workspace_dev >= the bytes above, 256-byte aligned,
 * valid for the farm's life.  offsets_out: int64 [2][nitems + 1], item = proposal * nchunks + chunk: row 0 where each
 * item's delta starts in delta_dev, row 1 where its Sigma (or diagonal) starts in sigma_dev, in doubles; entry nitems of
 * each row is that buffer's length.  A chunk's items are contiguous, proposal after proposal.  Launch choices and
 * look-ahead follow psoap_chunk.reserved as the gradient graph's do, so that with the reserved value set the outputs
 * depend neither on nbranch nor on how the chunks are partitioned over ranks. */
size_t psoap_farm_predict_workspace_bytes(const psoap_farm *farm, int nbranch, const int64_t *m, int sigma_mode);
int psoap_farm_predict_attach(psoap_farm *farm, int nbranch, const int64_t *m, const double *const *grids_dev,
                              int sigma_mode, void *workspace_dev, size_t workspace_bytes, int64_t *offsets_out);
/* p_dev: [nprop][n_params] contiguous, as psoap_farm_lnprob.  Per item: delta = C K^-1 (fl - mu_GP), the components
 * stacked [ncomp * m] (the caller adds the component means), Sigma row-major [ncomp m][ncomp m] or its diagonal, and
 * the item's record in results_dev [nprop][nchunks] (lnlike, logdet, quad, info of the chunk's data block).  Every output
 * of an item is NaN when its sentinel fired (|v| >= c, a negative GP value; lnlike -inf, info 0) or info != 0; other
 * items are unaffected.  No floating-point atomics: the outputs are bit-identical from call to call.  PSOAP_ERR_ARG
 * before psoap_farm_predict_attach. */
int psoap_farm_predict(psoap_farm *farm, const double *p_dev, double *delta_dev, double *sigma_dev,
                       psoap_result *results_dev, void *stream);

/* ---- measurement helpers ----------------------------------------------------------------------------- */
/* Register-resident DMMA.8x8x4 loop on all SMs: measured FP64 tensor-pipe peak in TFLOP/s (synchronous). */
int psoap_fp64_peak_tflops(double *tflops_out);
/* Times the dominant kernel (the DMMA trailing update, csrc/gemm.cuh syrk3_kernel)
 * alone: `reps` launches of the rank-K update (K a multiple of 128, up to 512 in the factorisation) of an m x m
 * lower triangle, CUDA events on the launching stream.  flops_per_launch is the algorithmic count K m (m + 1)
 * (DSYRK convention; the upper halves of the diagonal tiles are computed but not counted). Synchronous. */
int psoap_bench_syrk(int64_t m, int K, int reps, double *avg_ms_out, double *flops_per_launch_out);
/* The same launch with the partial last round of tiles dealt out as quarter tiles (tail_split = 1) or whole
 * (0): psoap_bench_syrk uses the library's shipped setting (0, see api.cu g_tail_split for the measurements). */
int psoap_bench_syrk_split(int64_t m, int K, int reps, int tail_split, double *avg_ms_out, double *flops_per_launch_out);
/* The likelihood's INTERNAL fill (csrc/fill.cuh fill_lower_kernel) written into a caller-provided matrix, for the
 * entry-wise parity tests against psoap/matrix_functions.pyx:125-144 (+ covariance.py:322, data.py:40-63).
 * W_dev: column-major [Np, ld], Np = N rounded up to 128, ld >= Np and even; data index i lives at i + (Np - N);
 * only the lower triangle is written (identity in the padding).  rvec_dev [Np] receives fl - mu_GP.
 * epoch_dev/vel_dev NULL: lwl_f/g/h are already shifted per-component vectors; otherwise lwl_f is the base vector and
 * vel_dev [ncomp, n_epochs] the velocity table, the Doppler shift being fused into the fill.  Synchronous. */
int psoap_debug_fill_lower(int ncomp, int64_t N, const double *lwl_f_dev, const double *lwl_g_dev,
                           const double *lwl_h_dev, const int32_t *epoch_dev, const double *vel_dev, int n_epochs,
                           const double *fl_dev, const double *sigma_dev, const double *amp, const double *l,
                           double mu_GP, double *W_dev, int64_t ld, double *rvec_dev, void *stream);
/* Times a fill kernel alone on the caller's shifted device vectors: kind 0 = the internal lower-triangle fill
 * (4 N^2 algorithmic bytes), kind 1 = the operator-surface fill_V11_* (8 N^2 bytes).  Synchronous. */
int psoap_bench_fill(int kind, int ncomp, int64_t N, const double *lwl_f_dev, const double *lwl_g_dev,
                     const double *lwl_h_dev, const double *amp, const double *l, int reps, double *avg_ms_out);
/* Host-side replay of the trailing-update tile enumeration (csrc/gemm.cuh SyrkSrc::decode; no device work): the
 * (row tile r, 64-column tile jrel) of every tile of a launch over R row tiles for part 0 (all), 1 (first ncol1
 * column tiles of every row) or 2 (the rest).  Returns the tile count, -1 if cap is too small. */
int psoap_debug_syrk_tiles(int R, int part, int ncol1, int *rows_out, int *cols_out, int cap);
/* Number of kernels launched by this library since load (for bench.py's gpu_launches). */
int64_t psoap_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* PSOAP_B200_H */
