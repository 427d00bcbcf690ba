/*
 * ba_b200.h -- C ABI of the B200-native bundle-adjustment engine (libba_b200.so).
 *
 * Drop-in boundary for the perspective-camera Levenberg-Marquardt refinement of the reference
 * repository takah29/3d-reconstruction-from-multi-view-exp, file lib/bundle_adjustment.py
 * (class BundleAdjuster).  The reference is pure Python and has no FFI of its own; these are
 * the entry points a binding for that class needs (SURVEY.md section 8b, last row), and each
 * one cites the reference lines it replaces.  INTEGRATION.md shows the ctypes stub.
 *
 * Conventions
 *   - plain C types only; every array is float64 unless stated; the caller owns all buffers;
 *   - `mem` says where the caller's buffers live: BA_MEM_HOST or BA_MEM_DEVICE (a raw device
 *     pointer, e.g. torch.Tensor.data_ptr());
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream); all work of
 *     a call is enqueued on it; calls that return values to host memory synchronise it;
 *   - every function returns a ba_status; ba_last_error() gives the message of the last
 *     failure on the calling thread;
 *   - state is held in the *normalised gauge frame* of the reference (camera 0 = identity at
 *     the origin, baseline component = +-1; lib/bundle_adjustment.py:208-240).  The O(N)
 *     normalise / denormalise steps run either on the host side of the boundary (ba_set_state /
 *     ba_get_state take and return the normalised frame) or on the device
 *     (ba_set_state_global / ba_get_state_global take and return the caller's frame).
 *   - one engine per process and GPU.  Points may be sharded over several engines (one per
 *     rank); the camera block is replicated and two sums per inner solve run over the ranks:
 *     by the library's own kernels over NVLink peer memory (ba_comm_*), or by the host
 *     all-reducing two device buffers (ba_reduce_buffer / ba_cost_buffer) between the phases.
 */
#ifndef BA_B200_H
#define BA_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BA_B200_VERSION 1

typedef struct ba_engine ba_engine;

typedef enum ba_status {
  BA_OK = 0,
  BA_ERR_INVALID = 1,   /* bad argument            -> ValueError   (reference :28, :232)   */
  BA_ERR_CUDA = 2,      /* CUDA runtime failure     -> RuntimeError                         */
  BA_ERR_SINGULAR = 3,  /* singular point block     -> LinAlgError  (reference :128, :146)  */
  BA_ERR_STATE = 4,     /* call out of order        -> RuntimeError                         */
  BA_ERR_NO_DEVICE = 5, /* no CUDA device           -> RuntimeError (there is no CPU path)  */
  BA_ERR_STALL = 6,     /* inner LM loop exceeded max_retries -> RuntimeError (the reference
                           loops forever, :118; documented deviation)                       */
  BA_ERR_COMM = 7,      /* a peer rank did not answer within the spin limit -> RuntimeError  */
  BA_ERR_BARRIER = 8    /* a grid-wide barrier inside one kernel timed out  -> RuntimeError  */
} ba_status;

enum { BA_MEM_HOST = 0, BA_MEM_DEVICE = 1 };
enum { BA_AXIS_X_RIGHT = 0, BA_AXIS_X_UP = 1 }; /* reference :23-33, :62-72 */
enum { BA_STATE_CURRENT = 0, BA_STATE_TRIAL = 1 };

/* Problem description (constructor arguments of the reference class, :11-21, in
 * observation-list form). */
typedef struct ba_problem {
  int64_t n_points;     /* points owned by this engine (a shard of the scene)                */
  int64_t n_obs;        /* visible (point, camera) pairs of those points                     */
  int32_t n_cams;       /* cameras (all of them; replicated on every shard)                  */
  int32_t axis;         /* BA_AXIS_*: which baseline component the gauge pins                */
  double f0;            /* image-coordinate scale (reference :18, :50)                       */
  int32_t dense;        /* 1: every point sees every camera, obs o = point*n_cams + camera   */
  int32_t device;       /* CUDA device ordinal                                               */
} ba_problem;

/* Levenberg-Marquardt control block, mirrored from device memory (reference :100-195). */
typedef struct ba_lm_state {
  double E;             /* cost of the current (accepted) state                              */
  double E_trial;       /* cost of the last trial state                                      */
  double c;             /* Marquardt damping factor (:100, :165, :195)                       */
  double delta;         /* |E_trial - E| of the last accepted iteration (:186)               */
  double scale_factor;  /* :79                                                               */
  double delta_tol;     /* :80                                                               */
  int32_t count;        /* accepted iterations so far (:185)                                 */
  int32_t max_iter;     /* :81                                                               */
  int32_t solves;       /* inner solves so far                                               */
  int32_t iter_solves;  /* inner solves of the iteration in progress                         */
  int32_t need_linearize; /* 1: next solve re-linearises (after an accept)                   */
  int32_t accepted;     /* 1: the last decide() accepted the trial                           */
  int32_t done;         /* 1: terminated (:191)                                              */
  int32_t status;       /* ba_status raised on the device (singular block, stall)            */
  int32_t chol_fail;    /* 1: last reduced system was not positive definite (step rejected)  */
  int32_t max_retries;  /* cap on inner solves per iteration                                 */
} ba_lm_state;

/* One record per accepted iteration (what the reference prints and logs, :175-188). */
typedef struct ba_iter_record {
  double E_prev;
  double E;
  double delta;
  double c;
  int32_t solves;
  int32_t count;
} ba_iter_record;

/* ---- life cycle ------------------------------------------------------------------- */
int ba_version(void);
const char* ba_last_error(void);
int ba_device_count(void);
/* BundleAdjuster.__init__ (:11-75) after host-side gauge normalisation. */
int ba_create(const ba_problem* problem, ba_engine** out);
int ba_destroy(ba_engine* e);

/* Observations (:36-37, :56-60) as CSR by point: obs_ptr[n_points+1], obs_cam[n_obs] (may be
 * NULL when problem.dense), obs_xy[n_obs][2].  Builds the camera-major index on the device. */
int ba_set_observations(ba_engine* e, const int64_t* obs_ptr, const int32_t* obs_cam,
                        const double* obs_xy, int mem, void* stream);
/* Dense observations exactly as the reference constructor receives them (`x`, :36-37): element
 * (point j, camera i, c) lies at x[j * stride_pt + i * stride_cam + c] (strides in doubles).  Two
 * layouts are taken: one point-major block (stride_pt = 2 n_cams, stride_cam = 2) and one
 * camera-major block (stride_pt = 2, stride_cam = 2 n_points) -- what both reference scripts pass,
 * np.stack(x_list).transpose(1, 0, 2) (euclidiean_reconstruction.py:54).  The block is copied as it
 * lies in memory and re-ordered to point-major on the device, so the host never makes the
 * contiguous copy.  Any other stride pattern returns BA_ERR_INVALID (copy on the host first). */
int ba_set_observations_dense(ba_engine* e, const double* x, int64_t stride_pt, int64_t stride_cam,
                              int mem, void* stream);
/* State in the normalised frame: X[n_points][3], R[n_cams][3][3], t[n_cams][3], f[n_cams],
 * u[n_cams][2]  (:40-48).  Any pointer may be NULL to leave that part untouched. */
int ba_set_state(ba_engine* e, const double* X, const double* R, const double* t,
                 const double* f, const double* u, int mem, void* stream);
int ba_get_state(ba_engine* e, int which, double* X, double* R, double* t, double* f, double* u,
                 int mem, void* stream);
/* The same in the CALLER's frame, with the gauge handled on the device (SURVEY.md 8f row 1):
 * ba_set_state_global takes init_X / init_R / init_t as the constructor receives them (:11-21),
 * keeps camera 0's pose and the baseline length (:23-33) and stores the normalised state
 * (_transform_to_normalize_coodinates, :208-240, incl. its signed divisor);
 * ba_get_state_global returns state `which` transformed back (:242-258) with K assembled
 * from f, u, f0 (:283-289): X[n_points][3], K[n_cams][3][3], R[n_cams][3][3], t[n_cams][3]. */
int ba_set_state_global(ba_engine* e, const double* X, const double* R, const double* t,
                        const double* f, const double* u, int mem, void* stream);
int ba_get_state_global(ba_engine* e, int which, double* X, double* K, double* R, double* t,
                        int mem, void* stream);

/* ---- single kernels / phases (each cites what it replaces) --------------------------- */
/* _calc_reprojection_error (:666-677): local cost of the current state into the cost buffer
 * slot 0 (a partial sum when the scene is sharded). */
int ba_cost(ba_engine* e, int which, void* stream);
/* K1 + per-point and per-camera reductions: _calc_pqr, _calc_*_diff_pqr, _calc_d_P, _calc_d_F,
 * _calc_matE, _calc_matG (:103-116).  Unconditional. */
int ba_linearize(ba_engine* e, void* stream);
/* K2 + K3 for damping `c`: damp/invert V_j, Y_j, partial Schur products into the reduce
 * buffer (:120-143).  Unconditional. */
int ba_build_reduced(ba_engine* e, double c, void* stream);
/* K4 for damping `c` on the (all-reduced) reduce buffer: assemble, Cholesky, solve,
 * back-substitute, trial state and its local cost (:146-162).  Unconditional. */
int ba_solve_trial(ba_engine* e, double c, void* stream);

/* ---- the LM loop with its control flow on the device --------------------------------- */
/* optimize() prologue (:85-101): reset the control block, cost of the initial state. */
int ba_lm_begin(ba_engine* e, double scale_factor, double delta_tol, int max_iter,
                int max_retries, void* stream);
/* Phase 1 of an inner solve: (re-)linearise if flagged, build the partial reduced system.
 * Sharded runs all-reduce ba_reduce_buffer() afterwards. */
int ba_lm_phase_reduce(ba_engine* e, void* stream);
/* Phase 2: solve, trial state, local trial cost.  Sharded runs all-reduce ba_cost_buffer(). */
int ba_lm_phase_solve(ba_engine* e, void* stream);
/* Phase 3: accept / reject, damping schedule, termination (:164-195); commits the trial. */
int ba_lm_phase_decide(ba_engine* e, void* stream);
/* Copy the control block to the host (synchronises `stream`). */
int ba_lm_state_get(ba_engine* e, ba_lm_state* out, void* stream);
/* The same without stalling the stream: _post enqueues the copy into pinned slot `slot` (0 or 1)
 * and an event behind it, _wait blocks the host on that event only.  A loop that posts after
 * every decide and waits one solve later keeps the device one solve ahead of the host (every
 * kernel of a solve is a no-op once the control block says done). */
int ba_lm_state_post(ba_engine* e, int slot, void* stream);
int ba_lm_state_wait(ba_engine* e, int slot, ba_lm_state* out);
/* Run inner solves until one iteration is accepted or the loop terminates (single engine). */
int ba_lm_iterate(ba_engine* e, ba_lm_state* out, void* stream);
/* Whole optimize() loop (:102-195) for a single engine; records[0..*n_records) receive one
 * entry per accepted iteration (at most max_records). */
int ba_lm_run(ba_engine* e, double scale_factor, double delta_tol, int max_iter, int max_retries,
              ba_iter_record* records, int max_records, int* n_records, ba_lm_state* final_state,
              void* stream);
int ba_lm_records(ba_engine* e, ba_iter_record* records, int max_records, int* n_records,
                  void* stream);

/* ---- buffers the host all-reduces when points are sharded over ranks ----------------- */
/* Partial reduced system: [P (n_pad x n_pad) | U (n_cams x 81) | dF (n_cams x 9)] doubles. */
int ba_reduce_buffer(ba_engine* e, void** device_ptr, int64_t* n_doubles);
/* [cost slot 0 (current / initial), cost slot 1 (trial), 1.0 if a point block of this engine's
 * shard was singular in the trial solve else 0.0, pad] doubles.  A host that sums the trial cost
 * over the ranks sums elements 1..2 together, so that one rank's singular block (LinAlgError,
 * reference :128) stops every rank in the same solve. */
int ba_cost_buffer(ba_engine* e, void** device_ptr, int64_t* n_doubles);
/* Only one rank prints/logs; every rank must still hold the same U/dF: this marks whether
 * this engine's U/dF partials are to be counted (all ranks: 1). */

/* ---- sharded runs over NVLink peer memory (one process per GPU, <= 8 ranks of one box) --- */
/* The reference is a single process (SURVEY.md section 2.1: no parallelism of any kind); these
 * calls are the multi-GPU form of the sums at :135-143 and :674-676.  ba_comm_create allocates
 * this rank's exchange window (header + reduce buffer + one staging slot per rank), moves the
 * reduce buffer into it and returns an opaque blob (the window's CUDA IPC handle, its exchange
 * epochs and, in the last 8 bytes, 1 if the window is new / 0 if it is a recycled one that the
 * peers already map; BA_COMM_HANDLE_BYTES bytes).  Windows are kept for the life of the process and handed to
 * the next engine of the same shape, mappings included.
 * The host gathers the handles of all ranks in rank order (any transport; e.g.
 * torch.distributed.all_gather) and passes them to ba_comm_connect, then -- if any window is
 * new -- synchronises the ranks once (nobody may store into a window that is not mapped
 * everywhere yet).  From then on ba_lm_begin / ba_lm_phase_* / ba_lm_iterate / ba_lm_run sum the partial
 * reduced system and the costs over all ranks with the library's own kernels (peer stores,
 * deterministic rank-order addition); the host must NOT all-reduce the buffers as well. */
#define BA_COMM_HANDLE_BYTES 88
int ba_comm_create(ba_engine* e, int rank, int world, void* handle_out);
int ba_comm_connect(ba_engine* e, const void* handles /* world x BA_COMM_HANDLE_BYTES */);
/* Quiesce this engine's side of the exchange (drains its streams).  Optional: ba_destroy does the
 * same.  No rank-wide synchronisation is needed around destruction -- windows are never freed, and
 * an exchange can only start on a recycled window after every peer has left the previous one. */
int ba_comm_disconnect(ba_engine* e);
int ba_comm_world(ba_engine* e, int* rank, int* world);

/* ---- inspection (tests, ncu-free evidence); copies to host memory ------------------- */
typedef enum ba_buffer_id {
  BA_BUF_JP = 0,     /* [n_obs][8]  e0,e1, d e/dX (2x3)                    K1   */
  BA_BUF_JC = 1,     /* [n_obs][20] e0,e1, d e/d(f,u0,v0,t,w) (2x9)       K1   */
  BA_BUF_V = 2,      /* [n_points][6] xx,xy,xz,yy,yz,zz of matE (:519)     K2   */
  BA_BUF_GPT = 3,    /* [n_points][3] d_P (:429)                           K2   */
  BA_BUF_U = 4,      /* [n_cams][81] diagonal blocks of matG (:618), gauge rows zeroed */
  BA_BUF_GCAM = 5,   /* [n_cams][9]  d_F (:471), gauge entries zeroed            */
  BA_BUF_S = 6,      /* [n_pad][n_pad] reduced system after assembly / Cholesky (lower) */
  BA_BUF_DXI = 7,    /* [n_cams][9] camera step, zeros at the gauge entries (:146, :267) */
  BA_BUF_LINV = 8,   /* [n_points][6] inverse Cholesky factor of damped V_j     K2 */
  BA_BUF_Z = 9,      /* [n_points][3] L_j^-1 d_P_j                               K2 */
  BA_BUF_REDUCE = 10,/* the reduce buffer (see ba_reduce_buffer)                    */
  BA_BUF_COST = 11,  /* [4] see ba_cost_buffer                                      */
  BA_BUF_YT = 12     /* dense: [k_pad][n_pad] Y^T, the operand of the Schur product P = Yt^T Yt */
} ba_buffer_id;
int ba_buffer_size(ba_engine* e, int id, int64_t* n_doubles);
int ba_buffer_read(ba_engine* e, int id, double* host_out, int64_t n_doubles, void* stream);
/* Layout facts the host needs: padded order of the reduced system and its rhs row. */
int ba_reduced_layout(ba_engine* e, int32_t* n_pad, int32_t* n_full, int32_t* rhs_row);

/* ---- profiling helpers ------------------------------------------------------------ */
/* Number of kernels this library launched since ba_create (all engines of the process). */
int64_t ba_launch_count(void);
/* Device time (ms, CUDA events on `stream`) and launches of the named kernel group
 * accumulated while profiling is enabled; groups: "k1","k2","k3","k4","cost","other", and
 * nested inside k3 / k4: "syrk" (the DMMA kernel alone), "chol" (factor + solve), "comm" (the
 * peer-memory sums of a sharded run). */
int ba_profile_enable(ba_engine* e, int on);
int ba_profile_get(ba_engine* e, const char* group, double* total_ms, int64_t* launches);
int ba_profile_reset(ba_engine* e);
/* FP64 peak micro-benchmarks (register-resident loops): TFLOP/s.  use_dmma = 1: DMMA.8x8x4,
 * 0: DFMA, 2: both interleaved with equal FMA counts (do they share the FP64 datapath?), 100 + w:
 * the DFMA loop with w warps per SM (rate at low occupancy). */
int ba_fp64_peak(int device, int use_dmma, double* tflops);
/* How the 128-tile Schur SYRK / Cholesky trailing update gets its operands: 1 = TMA tensor copies +
 * mbarriers with a producer warp (cp.async.bulk.tensor, SASS UTMALDG), 0 = cp.async (LDGSTS; set
 * BA_SYRK_NO_TMA=1 for A/B timing, or the driver does not offer cuTensorMapEncodeTiled). */
int ba_syrk_feed(void);
/* 1 when this engine linearises matrix-free: a dense scene whose camera table fits shared memory
 * (<= 361 cameras) re-derives the Jacobian rows in K2a, the camera blocks, K2b and the point update
 * instead of storing them in K1 and reading them back (reference :309-427 evaluated where used);
 * 0 otherwise (sparse visibility, more cameras, or BA_NO_MATRIX_FREE=1).  ba_buffer_read of the
 * JP / JC rows still works: K1 writes them for that read. */
int ba_matrix_free(ba_engine* e);
/* Host-only (no device): plan the dense Schur product (K3) of an n_cams x n_points scene for a GPU
 * with num_sms SMs and `tile` = 64 or 128, verify that the work items cover every tile's K range
 * exactly once, and report the number of items / tiles and the modelled schedule length against
 * the perfectly balanced one (both in k-rows of a full tile per SM). */
int ba_syrk_plan_info(int n_cams, int64_t n_points, int tile, int num_sms, int* n_items, int* n_tiles,
                      double* makespan_rows, double* ideal_rows);
/* Host-only: the dense Schur product emulated on the INT8 tensor cores (Ozaki scheme II) -- the
 * moduli (moduli[0 .. *n_moduli), pass null to query the count) and b, the bits every scaled entry
 * keeps for a product over k_pad rows (largest b <= 53 with k_pad 2^(2b) < prod(moduli) / 2). */
int ba_syrk_emu_info(int64_t k_pad, int32_t* moduli, int* n_moduli, int* bits);
/* 1 when this engine's dense Schur product runs on the INT8 tensor cores (chosen at creation by size,
 * or by BA_SYRK_EMU=0|1), 0 when on the FP64 tensor cores or sparse. */
int ba_syrk_emulated(ba_engine* e);

/* ---- next to the path: batched re-projection ------------------------------------------- */
/* calc_projected_points (reference lib/camera.py:74-81, Camera.project_points :18-32): project
 * X[n_points][3] into every camera (K[n_cams][3][3] general, R camera-to-world, t centres);
 * out[n_cams][n_points][2] = (p/r, q/r).  No engine needed.  With BA_MEM_HOST the call copies
 * in, computes, copies out and synchronises `stream`; with BA_MEM_DEVICE all five pointers are
 * device pointers (out 16-byte aligned) and the call is asynchronous. */
int ba_project_points(int device, int64_t n_points, int32_t n_cams, const double* X, const double* K,
                      const double* R, const double* t, double* out, int mem, void* stream);

/* ---- before the path: projective-depth iteration, primary method --------------------------- */
/* _compute_projective_depth_primary_method (reference lib/perspective_camera_calibration.py:61-144,
 * with _compute_reprojection_error :44-58): x[n_points][n_images][3] are the rows (x/f0, y/f0, 1) of
 * _create_data_matrix (:35-41); z[n_points][n_images] receives the projective depths; errors (may be
 * NULL, else >= max_iter doubles) the reprojection error of every iteration (what the reference
 * prints, :141); *n_iter the number of iterations run (stops when E < tolerance or at max_iter,
 * :138-142).  2 <= n_images <= 64.  No engine needed; BA_MEM_HOST copies in and out. */
int ba_projective_depth_primary(int device, int64_t n_points, int32_t n_images, const double* x, double f0,
                                double tolerance, int max_iter, double* z, double* errors, int* n_iter,
                                int mem, void* stream);

/* _compute_projective_depth_dual_method (reference lib/perspective_camera_calibration.py:147-235) --
 * the method euclidiean_reconstruction.py:42 selects.  Same arguments as the primary entry point.
 * The reference builds an (n_images, n_points, n_points) array (:188); here every per-image N x N
 * eigenproblem is reduced to a 12 x 12 one (csrc/k7_projective_depth.cu), memory is O(n_images x
 * n_points).  The sign of each image's column of z -- which the reference leaves to LAPACK's
 * eigenvector convention (:206-215) -- is fixed by making the column's unit eigenvector sum
 * non-negative before the reference's row rule is applied; the Euclidean upgrade does not depend on
 * it.  max_iter < 1 runs one pass, like the reference.  2 <= n_images <= 64. */
int ba_projective_depth_dual(int device, int64_t n_points, int32_t n_images, const double* x, double f0,
                             double tolerance, int max_iter, double* z, double* errors, int* n_iter,
                             int mem, void* stream);

/* Tests only: register host buffers that the next ba_projective_depth_dual call fills with the
 * intermediates of its last pass (V4 [N][4], R60 [M][60], W12 [M][12], e [N][M], sums [2][M],
 * U4 [3M][4]); any may be NULL, all NULL switches the probe off. */
int ba_depth_dual_probe(double* V4, double* R60, double* W12, double* e, double* sums, double* U4);

/* factorization_method(W, n_rank=4) (reference lib/factorization.py:5-15), the step between the
 * projective depths and the Euclidean upgrade (lib/perspective_camera_calibration.py:533): rank-4
 * truncated SVD W ~ M S of the (n_rows x n_cols) matrix, n_rows = 3 n_images <= 192.  Wt is W
 * TRANSPOSED, [n_cols][n_rows] row-major (what the reference's `W.reshape(N, -1).T` is a view of);
 * M_out[n_rows][4] = the four leading left singular vectors, S_out[4][n_cols] = diag(Sigma) V^T,
 * sigma_out[4] (may be NULL) the singular values.  The reference's full SVD allocates an
 * n_cols x n_cols factor; here the Gram matrix W W^T goes through the FP64 tensor cores and only its
 * leading eigenspace is computed.  Singular vectors are defined up to sign, as in LAPACK. */
int ba_factorize_rank4(int device, int64_t n_cols, int32_t n_rows, const double* Wt, double* M_out,
                       double* S_out, double* sigma_out, int mem, void* stream);

/* The factorisation step of the affine self-calibrations (reference lib/affine_camera_calibration.py:
 * _get_observation_matrix :224-240 followed by np.linalg.svd at :21, :70, :154): every row of W
 * (n_rows = 2 n_images, one image coordinate each) is first centred over the points -- here every
 * column of the point-major array Wt [n_cols][n_rows], which is the reference's np.hstack(data_list)
 * as it lies in memory -- mean_out[n_rows] (may be NULL) receives the means (the image centroids t),
 * then the rank-4 factorisation above runs on the centred matrix; the callers use its three leading
 * components.  Same size limits and sign convention as ba_factorize_rank4. */
int ba_factorize_centred_rank4(int device, int64_t n_cols, int32_t n_rows, const double* Wt, double* mean_out,
                               double* M_out, double* S_out, double* sigma_out, int mem, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* BA_B200_H */
