/* mlb200.h — the thin C-ABI between the ML++ host classes and the B200 (sm_100a) CUDA kernels.
 *
 * The reference (romanwerpachowski/ML) has no FFI for its clustering path: the boundary a user sees
 * is the C++ class API (ML/Clustering.hpp:17-89, ML/EM.hpp:18-166, ML/KMeans.hpp:19-101) and the
 * pybind module (cppyml/clustering.cpp:75-184).  Those are kept unchanged by the host layer under
 * ml_b200/host/; this header is what that host layer calls, and what a replacement backend would
 * have to export.  Each entry point names the reference loop it replaces.
 *
 * Conventions
 *   - plain C, opaque handles, no exceptions, no torch/Eigen types;
 *   - every function returns 0 on success or an MLB_E* code; mlb_last_error() gives the text of the
 *     last failure on the calling thread;
 *   - matrices are column-major exactly like Eigen::MatrixXd: data is D x N (a point per column,
 *     D contiguous doubles per point), means/centroids are D x K, a covariance is D x D,
 *     responsibilities are N x K (element (i,k) at i + k*N);
 *   - a handle belongs to one host thread at a time;
 *   - everything is FP64; labels are unsigned int as in the reference;
 *   - there is no CPU fallback: without a CUDA device every compute entry point fails with MLB_ECUDA.
 *
 * Sharding.  The N points are cut into fixed "chunks" (a function of N only) and the chunks into 8
 * contiguous virtual shards.  A context with G GPUs (G in {1,2,4,8}) gives 8/G consecutive virtual
 * shards to each GPU.  Per-chunk partial statistics are summed in a fixed order inside a virtual
 * shard, the 8 shard vectors are exchanged with ONE ncclAllGather per iteration and summed in the
 * fixed tree ((0+1)+(2+3))+((4+5)+(6+7)) on every GPU, so results are bit-identical across ranks and
 * across G.  (SURVEY.md §5, §8e.)
 */
#ifndef MLB200_H
#define MLB200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MLB_OK 0
#define MLB_EINVAL 1   /* bad argument (the reference throws std::invalid_argument / domain_error) */
#define MLB_ECUDA 2    /* CUDA runtime / driver failure, or no device */
#define MLB_ENCCL 3    /* NCCL failure */
#define MLB_ENOMEM 4   /* device or host allocation failed */
#define MLB_ESTATE 5   /* call sequence error (e.g. emit before any step) */

#define MLB_VIRTUAL_SHARDS 8
#define MLB_NCCL_UNIQUE_ID_BYTES 128

typedef struct mlb_ctx mlb_ctx;   /* a set of GPUs: all local (one process), or one rank of a job */
typedef struct mlb_data mlb_data; /* the point matrix, resident in HBM, sharded over the context */
typedef struct mlb_em mlb_em;     /* Gaussian-mixture EM state (ml::EM, ML/EM.hpp:168-187) */
typedef struct mlb_km mlb_km;     /* K-means state (ml::Clustering::KMeans, ML/KMeans.hpp:103-116) */

/* ---------------------------------------------------------------- library */

int mlb_version(void);                 /* 10000*major + 100*minor + patch */
const char* mlb_last_error(void);      /* thread-local, never NULL */
int mlb_device_count(int* count);      /* cudaGetDeviceCount */

/* Diagnostic: evaluates the kernels' own FP64 exp (arguments <= 0, ml_b200/csrc/fastmath.cuh) for n host
 * values on device 0, so that tests can bound its error against libm.  Replaces std::exp of EM.cpp:206. */
int mlb_selftest_exp(const double* x, int64_t n, double* out);

/* Diagnostic: the FP64 peaks of `device` in TFLOP/s, measured now with two dependent-chain micro-kernels that saturate
 * the SM's FP64 unit: mma.sync.m8n8k4.f64 (DMMA, the instruction the kernels issue) and DFMA.  About 50 ms.  bench.py
 * uses the DMMA figure as its roofline denominator (MEASURED_PEAKS.json has no FP64 entry). */
int mlb_selftest_fp64_peak(int device, double* dmma_tflops, double* dfma_tflops);

/* ---------------------------------------------------------------- context */

/* One process driving n_devices local GPUs (n_devices in {1,2,4,8}); devices == NULL means
 * 0..n_devices-1.  With n_devices > 1 the GPUs are joined by ncclCommInitAll. */
int mlb_ctx_create(const int* devices, int n_devices, mlb_ctx** out);

/* One process per GPU (torchrun style).  Rank 0 calls mlb_nccl_unique_id() and ships the 128
 * bytes to the other ranks (any side channel: torch.distributed broadcast, a file, MPI);
 * every rank then calls mlb_ctx_create_rank with the same id.  world in {1,2,4,8}. */
int mlb_nccl_unique_id(void* out128);
int mlb_ctx_create_rank(int device, int rank, int world, const void* nccl_unique_id128, mlb_ctx** out);

int mlb_ctx_destroy(mlb_ctx* ctx);
int mlb_ctx_world(const mlb_ctx* ctx, int* world, int* n_local, int* first_rank);

/* Sum of `local` over the ranks of a one-process-per-GPU job (one 8-byte ncclAllGather; every rank must call it);
 * in a single-process context *total = local.  The host classes use it to learn the total point count when every
 * rank passes its own rows to fit(). */
int mlb_ctx_sum_int64(mlb_ctx* ctx, int64_t local, int64_t* total);

/* Blocks until every local stream of the context is idle. */
int mlb_ctx_synchronize(mlb_ctx* ctx);

/* Elapsed device time helpers for benchmarks: CUDA events on the context's own streams
 * (torch.cuda.Event cannot see them).  mlb_ctx_timer_stop returns the MAX over local GPUs, in ms. */
int mlb_ctx_timer_start(mlb_ctx* ctx);
int mlb_ctx_timer_stop(mlb_ctx* ctx, double* elapsed_ms);

/* The half-open global point range [begin, end) that `rank` of `world` holds for a problem of
 * n_total points.  A pure function (no context needed). */
int mlb_shard_range(int64_t n_total, int world, int rank, int64_t* begin, int64_t* end);

/* ---------------------------------------------------------------- data */

/* Copies the host matrix (column-major D x n, outer stride ld >= d doubles) into HBM.
 * Single-process contexts take the whole matrix (n == n_total) and scatter it over their GPUs.
 * Rank contexts take the rank's own range of mlb_shard_range(n_total, world, rank).
 * Replaces nothing in the reference (its data never leaves host memory); the reference's
 * `fit(Eigen::Ref<const Eigen::MatrixXd> data)` argument is what is passed here (EM.cpp:91). */
int mlb_data_upload(mlb_ctx* ctx, const double* x, int64_t n, int64_t n_total, int d, int64_t ld, mlb_data** out);

/* Wraps points that already live in device memory of a 1-GPU context (no copy; the caller keeps
 * ownership and must keep the buffer alive).  Point-contiguous, D doubles per point. */
int mlb_data_wrap_device(mlb_ctx* ctx, const double* x_device, int64_t n, int d, mlb_data** out);

/* Synthetic benchmark data generated in HBM (SURVEY.md §8d): a K-component Gaussian mixture with
 * means U[-spread, spread]^D, covariances A A^T / D + 0.5 I, Dirichlet-like weights; point i is a
 * pure function of (seed, i) (Philox4x32-10 counter RNG), so every G sees identical data.
 * true_means (D x k_true), if not NULL, receives the generating means. */
int mlb_data_generate_gmm(mlb_ctx* ctx, int64_t n_total, int d, int k_true, uint64_t seed, double spread,
                          double* true_means, mlb_data** out);

/* Copies `count` points starting at GLOBAL index `begin` back to the host (column-major D x count).
 * Rank contexts can only read their own range. */
int mlb_data_download(mlb_data* data, int64_t begin, int64_t count, double* out);

int mlb_data_shape(const mlb_data* data, int64_t* n_total, int64_t* n_local, int* d);
int mlb_data_free(mlb_data* data);

/* standardise_features of the reference's Python package (cppyml/cppyml/utils.py:8-28) on the first local GPU: every
 * dimension minus its mean and, when n > 1, divided by its BIASED standard deviation (a zero deviation divides by zero,
 * as numpy does).  x and out are column-major D x n (a point per column) with outer strides ld, ld_out >= d; they may
 * be the same buffer.  Sums are pairwise trees in a fixed order (numpy's accuracy, bitwise reproducible). */
int mlb_standardise_features(mlb_ctx* ctx, const double* x, int64_t n, int d, int64_t ld, double* out, int64_t ld_out);

/* ---------------------------------------------------------------- initialisers (ML/Clustering.cpp) */

/* The distance pass of KPP::init (Clustering.cpp:42-51), kept incrementally: a per-point vector `nearest`
 * (squared distance to the nearest centroid chosen so far) stays resident next to the points and
 *     nearest_i <- min(nearest_i, (x_i - centroid).squaredNorm())
 * is applied for the newest centroid (D doubles); `first` != 0 starts from +infinity, i.e. leaves the plain
 * squared distance to this centroid.  The values equal the ones the reference recomputes from scratch over
 * all chosen centroids (a minimum does not depend on the order), at O(N D) per new centroid instead of
 * O(N n D).  nearest_out (may be NULL: the pass is then only enqueued) receives the vector: n_total
 * doubles, or the rank's own range in a rank context.  The draw itself (std::discrete_distribution over these weights, Clustering.cpp:55-56)
 * stays on the host so that the caller's PRNG stream is the reference's. */
int mlb_data_kpp_update(mlb_data* data, const double* centroid, int first, double* nearest_out);
/* Number of kernels the library launched on this object after its creation (the seeding passes). */
int mlb_data_launch_count(const mlb_data* data, int64_t* launches);

/* ---------------------------------------------------------------- Gaussian-mixture EM (ML/EM.cpp) */

/* Any K >= 1; D <= 128 (MLB_EINVAL beyond: the parameter refresh factorises a D x D covariance inside one SM). */
int mlb_em_create(mlb_ctx* ctx, mlb_data* data, int k, mlb_em** out);
int mlb_em_destroy(mlb_em* em);

/* EM::calculate_sample_covariance (EM.cpp:265-272): unbiased covariance of all points, D x D. */
int mlb_em_sample_covariance(mlb_em* em, double* cov_out);

/* Loads theta = (means D x K, covariances K blocks of D x D, mixing weights K) and runs
 * EM::process_covariances (EM.cpp:274-287: Cholesky, inverse, sqrt|Sigma|) on the device. */
int mlb_em_set_params(mlb_em* em, const double* means, const double* covariances, const double* weights);

/* EM::maximisation_step (EM.cpp:221-263) from host responsibilities (N x K column-major; rank
 * contexts pass their own rows, n_local x K with leading dimension n_local) — the
 * `maximise_first` start (EM.cpp:120-125). */
int mlb_em_mstep_from_responsibilities(mlb_em* em, const double* resp, int64_t ld);

/* The same from hard assignments (n_total labels in [0, K), or the rank's own range): the M-step of the
 * one-hot responsibilities ClosestCentroid::init writes (Clustering.cpp:72-89, `maximise_first` start),
 * without the N x K host matrix.  The labels are what mlb_km_assign / mlb_km_get_labels give for the
 * initial centroids (same strict <, lowest index wins). */
int mlb_em_mstep_from_labels(mlb_em* em, const unsigned int* labels);

/* One iteration of the hot loop (EM.cpp:143-147): expectation_step with the current theta_t, then
 * maximisation_step, fused on the device.  Returns the log-likelihood of theta_t (mean per point,
 * EM.cpp:211).  theta_t is kept for mlb_em_emit. */
int mlb_em_step(mlb_em* em, double* log_likelihood);

/* Asynchronous variant for benchmarks: enqueues `steps` iterations without reading anything back.
 * log_likelihoods (steps entries, may be NULL) is filled when the call returns (one sync at the end). */
int mlb_em_run_steps(mlb_em* em, int steps, double* log_likelihoods);

/* Current theta: means D x K, covariances K x (D x D), weights K.  Any pointer may be NULL. */
int mlb_em_get_params(mlb_em* em, double* means, double* covariances, double* weights);

/* process_covariances outputs for the current theta: inverse covariances K x (D x D) as computed by
 * LLT::solve(Identity) and sqrt|Sigma_k| (EM.cpp:280-285); used by the host-side
 * EM::assign_responsibilities (EM.cpp:176-188).  Any pointer may be NULL. */
int mlb_em_get_precisions(mlb_em* em, double* inverse_covariances, double* sqrt_determinants);

/* The E-step of the LAST mlb_em_step again, at the saved theta_t, writing what the reference
 * leaves in responsibilities_ (EM.cpp:213-218; N x K column-major with leading dimension ld) and
 * labels_ (EM.cpp:289-304; argmax, first maximum wins).  Either pointer may be NULL.
 * Rank contexts receive their own rows. */
int mlb_em_emit(mlb_em* em, double* resp_out, int64_t ld, unsigned int* labels_out);

/* The same for the GLOBAL point range [begin, begin + count) only (resp_out is count x K with leading
 * dimension ld, labels_out has count entries).  Rank contexts can only emit rows they hold. */
int mlb_em_emit_range(mlb_em* em, int64_t begin, int64_t count, double* resp_out, int64_t ld, unsigned int* labels_out);

/* EM::assign_responsibilities (EM.cpp:176-188) for m points at once, with the CURRENT parameters (after a
 * fit: the post-fit ones, as in the reference): x is column-major D x m with outer stride ld_x >= D, on
 * the host; resp_out (may be NULL) is m x K column-major with leading dimension ld_out >= m; labels_out
 * (may be NULL) is the argmax of each row (first maximum wins).  Runs on the first local GPU. */
int mlb_em_predict(mlb_em* em, const double* x, int64_t m, int64_t ld_x, double* resp_out, int64_t ld_out, unsigned int* labels_out);

/* Per-launch device timing of the dominant kernel (the fused E+M kernel) for roofline reports:
 * CUDA events recorded on the launching stream around each launch while enabled (at most 4096
 * launches are kept).  mlb_em_kernel_time_ms synchronises and returns the summed duration and the
 * number of launches measured on the first local GPU. */
int mlb_em_set_kernel_timing(mlb_em* em, int enabled);
int mlb_em_kernel_time_ms(mlb_em* em, double* total_ms, int64_t* launches);

/* Which device path the last step used: 1 = fused DMMA E+M kernel, 2 = split E / M kernels (both in feature space
 * about the data mean), 3 = direct-difference E / M kernels (per-component centring, as EM.cpp:205-207,246-248). */
int mlb_em_last_path(const mlb_em* em, int* path);
/* How many steps of this object took the direct-difference kernels so far (bench.py reports it next to its timings). */
int mlb_em_direct_steps(const mlb_em* em, int64_t* steps);

/* Numerical domain of the feature-space kernels and the routing between the paths.  The feature-space kernels expand
 * the quadratic form about ONE shift c (the data mean); their error grows with kappa = max_k (mu_k - c)^T P_k (mu_k - c),
 * the squared distance of a component from the centre of the data in its own standard deviations (relative error
 * ~1e-16 kappa: 1e-13 for standardised data, 1e-8 for tight clusters 1e4 standard deviations apart).  The library
 * computes kappa with every parameter refresh and runs the next step on the direct-difference kernels whenever
 * kappa > 3e5 (about 1.5e-11 lost to cancellation), when D > 64 or K > 256 (shapes only those kernels take), or when forced.  Guaranteed domain: results
 * within 1e-9 of the reference wherever the reference itself is finite, for any K and D <= 128.
 * mlb_em_force_path: path = 3 always uses the direct kernels, 0 restores the automatic choice.
 * mlb_em_conditioning: kappa of the current parameters and the path the next step will take. */
int mlb_em_force_path(mlb_em* em, int path);
int mlb_em_conditioning(mlb_em* em, double* kappa_max, int* next_path);
/* Number of kernels the library launched on this object since creation (bench "gpu_launches"). */
int mlb_em_launch_count(const mlb_em* em, int64_t* launches);
/* Diagnostic: the kernel configuration chosen for this object from (D, K, chunk), so that tests can check which template
 * instances they run.  out[8] = {feature-space path (1 fused, 2 split, 0 none: only the direct kernels take the shape),
 * DP, KP, NT (8-component n-tiles of a group), MW (split M kernel: feature tiles per warp; 0 off the split path),
 * direct-kernel DP, direct-kernel NB (= DP / 8), points per chunk}.  Computes nothing. */
int mlb_em_kernel_config(const mlb_em* em, int out[8]);

/* ---------------------------------------------------------------- K-means (ML/KMeans.cpp) */

/* D <= 128 (MLB_EINVAL beyond); any K (centroids that do not fit one CTA's shared memory are processed in blocks, same
 * results).  D <= 64 runs the DMMA filter + exact refinement, wider points the reference's scan as written. */
int mlb_km_create(mlb_ctx* ctx, mlb_data* data, int k, mlb_km** out);
int mlb_km_destroy(mlb_km* km);

int mlb_km_set_centroids(mlb_km* km, const double* centroids /* D x K */);
int mlb_km_get_centroids(mlb_km* km, double* centroids /* D x K */);

/* KMeans::assignment_step (KMeans.cpp:167-178): swaps labels/old_labels, assigns every point to
 * its nearest centroid (direct-difference squared distance, strict <, lowest k wins), returns the
 * inertia and how many labels differ from the previous assignment (old_labels_ == labels_ of
 * KMeans.cpp:85 is n_changed == 0).  Also accumulates the per-cluster counts and sums that
 * mlb_km_update applies. */
int mlb_km_assign(mlb_km* km, double* inertia, int64_t* n_changed);

/* KMeans::update_step (KMeans.cpp:180-192): centroids <- per-cluster means of the last assignment
 * (an empty cluster goes to the origin), old centroids kept; returns ||C - C_old||_F^2
 * (KMeans.cpp:103). */
int mlb_km_update(mlb_km* km, double* centroid_shift_sq);

/* KMeans::assign_label (KMeans.cpp:153-165) for m points at once with the current centroids: x is
 * column-major D x m with outer stride ld_x >= D, on the host; labels_out[i] is the nearest centroid
 * (strict <, lowest index wins), sqdist_out[i] (may be NULL) its squared distance (x - c).squaredNorm().
 * Does not touch the labels, statistics or centroids of the fit.  Runs on the first local GPU. */
int mlb_km_predict(mlb_km* km, const double* x, int64_t m, int64_t ld_x, unsigned int* labels_out, double* sqdist_out);

/* labels_ of the last assignment; rank contexts receive their own range. */
int mlb_km_get_labels(mlb_km* km, unsigned int* labels);
int mlb_km_launch_count(const mlb_km* km, int64_t* launches);
/* Diagnostic: the kernel configuration chosen for this object.  out[8] = {DP, KP, KB (centroids per block), number of
 * centroid blocks, warps per CTA of the assignment kernel, exact (1: D > 64, the reference's scan), statistics kernel
 * (0 one-hot for K <= 32, 1 counting sort, 2 owner warps), points per chunk}.  Computes nothing. */
int mlb_km_kernel_config(const mlb_km* km, int out[8]);
/* As mlb_em_set_kernel_timing / mlb_em_kernel_time_ms, for the assignment kernel. */
int mlb_km_set_kernel_timing(mlb_km* km, int enabled);
int mlb_km_kernel_time_ms(mlb_km* km, double* total_ms, int64_t* launches);

/* ---------------------------------------------------------------- K-means start sets (KMeans::fit with number_initialisations_ > 1,
 * ML/KMeans.cpp:29-47; the 3-start fit of Benchmarks/bm_KMeans.cpp:39-45)
 *
 * The reference runs the starts of a multi-start fit one after the other.  An mlb_kms holds up to 4 starts ("sets": K centroids,
 * N labels, statistics each) on one resident data set and advances them in lockstep: one pass of the assignment kernel reads
 * every point once and scores it against all active sets, one reduction / exchange and one read-back serve all of them.  Per
 * set, labels, inertia, changed counts and centroids are bit for bit those of an mlb_km driven through the same calls.
 * `active` is a bit mask of the sets a call advances (bit s = set s); a start that has converged is simply left out of it. */
typedef struct mlb_kms mlb_kms;
/* 1 when n_sets (1..4) sets of k centroids fit one CTA's shared memory at this data's D (D <= 64), else 0: the caller then
 * runs the starts one at a time on an mlb_km (same results). */
int mlb_kms_supported(const mlb_data* data, int k, int n_sets);
int mlb_kms_create(mlb_ctx* ctx, mlb_data* data, int k, int n_sets, mlb_kms** out);
int mlb_kms_destroy(mlb_kms* kms);
int mlb_kms_set_centroids(mlb_kms* kms, int set, const double* centroids /* D x K */);
int mlb_kms_get_centroids(mlb_kms* kms, int set, double* centroids /* D x K */);
/* mlb_km_assign for every active set: inertia[s], n_changed[s] are written for active sets only (arrays of n_sets). */
int mlb_kms_assign(mlb_kms* kms, unsigned int active, double* inertia, int64_t* n_changed);
/* mlb_km_update for every active set: centroid_shift_sq[s] for active sets only. */
int mlb_kms_update(mlb_kms* kms, unsigned int active, double* centroid_shift_sq);
int mlb_kms_get_labels(mlb_kms* kms, int set, unsigned int* labels);
int mlb_kms_launch_count(const mlb_kms* kms, int64_t* launches);

#ifdef __cplusplus
}
#endif
#endif /* MLB200_H */
