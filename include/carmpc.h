/*
 * carmpc.h - C ABI of the B200 batch-evaluation library for CarMPC's hot path.
 *
 * The reference (ahmad12hamdan99/CarMPC) is pure Python and has no FFI of its own; the entry points
 * below are what a ctypes binding of its two hot loops replaces:
 *
 *   (A) terminal-set membership of a state      lib/terminal_set.py:107-113  (np.all(A @ point <= b))
 *       and its sampled LQR-rollout form         lib/terminal_set.py:53-59, 198-200
 *   (B) one condensed MPC QP per initial state  lib/mpc.py:318-335 (state feedback), :456-478 (output
 *       feedback), built from lib/matrix_gen.py:6-72, closed against lib/simulator.py:51-69 and the
 *       observer lib/mpc.py:439-448 for Monte-Carlo closed loops.
 *
 * Conventions
 *   - extern "C", plain pointers and sizes; no C++ or torch types.
 *   - Every function returns 0 on success and a negative carmpc_status on failure; nothing throws
 *     across the ABI.  carmpc_last_error() returns a thread-local message for the last failure.
 *   - Pointers named d_* are DEVICE pointers owned by the caller; h_* are HOST pointers.
 *     `stream` is a cudaStream_t passed as void* (NULL = legacy default stream).
 *   - Handles are opaque, created and destroyed by the library, bound to the CUDA device that was
 *     current at creation, and may be used from one host thread at a time.
 *   - Sample grids are structure-of-arrays float64: four arrays x, y, psi, v of n elements.
 *   - Membership results are bitsets: bit (i & 31) of word (i >> 5) is sample i; the unused high
 *     bits of the last word are zero.
 */
#ifndef CARMPC_H
#define CARMPC_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum carmpc_status {
    CARMPC_OK = 0,
    CARMPC_ERR_INVALID = -1,   /* bad argument (null pointer, size out of range, bad handle kind) */
    CARMPC_ERR_CUDA = -2,      /* a CUDA runtime call failed; message has the CUDA error string  */
    CARMPC_ERR_NUMERIC = -3,   /* host setup failed (matrix not positive definite, ...)          */
    CARMPC_ERR_UNSUPPORTED = -4
} carmpc_status;

/* QP status codes written per sample */
#define CARMPC_QP_SOLVED 0
#define CARMPC_QP_INFEASIBLE 1 /* primal infeasible: the state is outside the region of attraction; the
                                  reference raises OutsideTheRegionOfAttractionError (lib/mpc.py:336-338) */
#define CARMPC_QP_MAX_ITER 2

const char* carmpc_last_error(void);
const char* carmpc_version(void);
void carmpc_destroy(void* handle);

/* ------------------------------------------------------------------------------------------------
 * (A) terminal-set membership
 * ---------------------------------------------------------------------------------------------- */

/* H-representation {x : A x <= b}.  h_Ab: rows x 5 row-major [a0 a1 a2 a3 | b] - exactly the layout of
 * terminal_sets/<env>_<goal>.npy (lib/terminal_set.py:206-210, lib/mpc.py:101-102).  rows <= 512. */
int carmpc_polytope_create(const double* h_Ab, int rows, void** handle);

/* Membership of n samples: bit i = all_r( fma(a3,v, fma(a2,psi, fma(a1,y, a0*x))) <= b ).
 * Replaces the triple loop lib/terminal_set.py:107-113.
 *   mode 0: every row evaluated in float64.
 *   mode 1: float32 screen with a rigorous error bound, float64 re-evaluation of every row whose
 *           float32 margin is inside the bound.  Same bits as mode 0 by construction.
 * d_bits: ceil(n/32) words.  d_count (nullable): number of members, int64, overwritten. */
int carmpc_membership_bitset(void* polytope, const double* d_x, const double* d_y, const double* d_psi,
                             const double* d_v, int64_t n, uint32_t* d_bits, int64_t* d_count, int mode,
                             void* stream);

/* Profile-guided row order: evaluates a strided subsample of the given samples and re-orders the rows so that the
 * ones that reject most samples come first (whole-warp early exit).  Results never depend on the order.
 * carmpc_membership_bitset does this by itself on its first call with n >= 2^20. */
int carmpc_polytope_tune(void* polytope, const double* d_x, const double* d_y, const double* d_psi, const double* d_v,
                         int64_t n, void* stream);

/* The same test on an implicit tensor grid (the reference builds its grid from linspace / arange,
 * lib/terminal_set.py:96-106): sample i has multi-index (i0, i1, i2, i3) in C order over
 * (n0, n1, n2, n3) and coordinate axis_k[i_k]; axis_to_state[k] in {0,1,2,3} says which state
 * component (x, y, psi, v) axis k carries.  h_axes: the four axes concatenated (host). */
int carmpc_membership_grid(void* polytope, const double* h_axes, const int32_t dims[4],
                           const int32_t axis_to_state[4], uint32_t* d_bits, int64_t* d_count, void* stream);

/* Host-buffer convenience (end-to-end path): pinned or pageable host SoA arrays in, host bitset out;
 * the copies are chunked and overlapped with the kernel on internal streams. */
int carmpc_membership_bitset_host(void* polytope, const double* h_x, const double* h_y, const double* h_psi,
                                  const double* h_v, int64_t n, uint32_t* h_bits, int64_t* h_count, int mode);

/* LQR-rollout form of the terminal set.  e_0 = p - goal, e_{t+1} = A_k e_t; state rows
 * Acon e_t <= bcon for t = 0..k_steps; input rows Ain e_t <= bin at t = 0 only
 * (input_check_mode 0, what lib/terminal_set.py:198-203 does) or at every step (mode 1).
 * h_Ak: 4x4 row-major; h_Acon: s x 4, h_bcon: s (already shifted to the goal, unit-norm rows as
 * the reference's polytope construction makes them); h_Ain: rin x 4, h_bin: rin. */
int carmpc_rollout_create(const double* h_Ak, const double* h_Acon, const double* h_bcon, int s,
                          const double* h_Ain, const double* h_bin, int rin, const double* h_goal,
                          int k_steps, int input_check_mode, void** handle);

/* The float32 screen of a rollout handle evaluates the EXPANDED rows g = a_r A_k^t (k_steps + 1 copies of the state rows,
 * 140 rows for the shipped sets), most of which are redundant (the reference reduces the same set to ~42 rows,
 * lib/terminal_set.py:203).  carmpc_rollout_get_rows returns the expanded rows as this handle built them (row-major
 * [rows][5] = g (4), b' in absolute coordinates; returns the row count, 0 if the handle has no screen; h_rows may be
 * NULL).  carmpc_rollout_reduce_screen keeps only rows h_kept for the screen; every other row d needs a redundancy
 * certificate: n_dual (row index, weight >= 0) pairs over kept rows with  g_d = sum w_k g_k  and  sum w_k b_k <= b_d
 * (the dual solution of  max g_d . p  over the kept rows).  The library only CHECKS the certificates (in long double,
 * against its own rows) and widens the screen's acceptance band by what they leave open; samples inside the band are
 * decided by the float64 step-by-step rollout as before, so results never depend on the reduction. */
int carmpc_rollout_get_rows(void* rollout, double* h_rows, int capacity);
int carmpc_rollout_reduce_screen(void* rollout, const int32_t* h_kept, int n_kept, const int32_t* h_dual_idx,
                                 const double* h_dual_w, int n_dual);

/* d_first_violation (nullable): int32 per sample, first step t at which a row is violated, -1 if none. */
int carmpc_rollout_bitset(void* rollout, const double* d_x, const double* d_y, const double* d_psi,
                          const double* d_v, int64_t n, uint32_t* d_bits, int32_t* d_first_violation,
                          int64_t* d_count, void* stream);

/* Host-buffer form of the rollout test (same chunked, overlapped pipeline as the H-rep one). */
int carmpc_rollout_bitset_host(void* rollout, const double* h_x, const double* h_y, const double* h_psi,
                               const double* h_v, int64_t n, uint32_t* h_bits, int32_t* h_first_violation,
                               int64_t* h_count);

/* Tuning hook for the streaming scans (polytope or rollout handle): staging geometry of the bulk-async kernel -
 * threads per CTA, ring slots per warp, 128-sample tiles per ring slot.  Results never depend on it; combinations the
 * library was not built with return CARMPC_ERR_UNSUPPORTED.  Default 128 / 2 / 1. */
int carmpc_scan_staging(void* handle, int threads_per_cta, int ring_slots, int tiles_per_slot);

/* ------------------------------------------------------------------------------------------------
 * (A') one sample set sharded over the GPUs of a box (BASELINE config 2: "a 10^8-point grid sharded
 *      across 1/2/4/8 B200"; north_star: the membership bitsets are gathered over NVLink)
 *
 * Every rank owns a WINDOW: the full bitset of the n_total samples (double-buffered), one member count per rank and
 * one step flag per rank, in peer-mappable device memory.  A sharded scan stores the words of its shard straight into
 * the windows of ALL ranks from inside the scan kernel (one 128-byte store per 1024 samples and destination, over
 * NVLink), then a one-warp kernel publishes the rank's count and flag and waits for every other rank's: there is no
 * separate all-gather.  One process per GPU: exchange the 64-byte handles of carmpc_shard_export with any host
 * mechanism (torch.distributed all_gather in carmpc_b200/sharding.py) and pass all `world` of them, in rank order, to
 * carmpc_shard_connect.  Several ranks inside one process: carmpc_shard_connect_local.
 * All ranks must call the *_sharded functions the same number of times (they are collective steps).
 * ---------------------------------------------------------------------------------------------- */
int carmpc_shard_create(int rank, int world /* <= 8 */, int64_t n_total, void** handle);
int carmpc_shard_export(void* shard, unsigned char* h_ipc_handle64);
int carmpc_shard_connect(void* shard, const unsigned char* h_ipc_handles /* world x 64 bytes, rank order */);
int carmpc_shard_connect_local(void* shard, void* const* peer_shards /* world handles, entry [rank] ignored */);

/* Membership of this rank's shard.  group_stride = 1: the n_local samples are [first_sample, first_sample + n_local)
 * of the set, first_sample a multiple of 32 (contiguous shards).  group_stride = s > 1: the k-th 1024-sample group of
 * the local arrays is group first_sample / 1024 + k s of the set, first_sample a multiple of 1024 (with s = world and
 * first_sample = 1024 rank the groups are dealt round-robin to the ranks: equal load whatever the cost profile of the
 * set is; only the last local group may be partial).  When the step has completed (stream order) the rank's window
 * holds the bitset of ALL n_total samples and *d_total_count (nullable, device int64) the member count over all ranks. */
int carmpc_membership_bitset_sharded(void* polytope, void* shard, const double* d_x, const double* d_y,
                                     const double* d_psi, const double* d_v, int64_t n_local, int64_t first_sample,
                                     int64_t group_stride, int mode, int64_t* d_total_count, int defer_wait, void* stream);
int carmpc_rollout_bitset_sharded(void* rollout, void* shard, const double* d_x, const double* d_y,
                                  const double* d_psi, const double* d_v, int64_t n_local, int64_t first_sample,
                                  int64_t group_stride, int64_t* d_total_count, int defer_wait, void* stream);
/* A collective step is scan (+ stores into every window), publish (count + flag, never blocks) and wait (blocks on the
 * device until every rank's flag has arrived).  defer_wait = 0: all three are enqueued by the *_sharded call (one
 * process per GPU).  defer_wait = 1: the call stops after publish and carmpc_shard_wait enqueues the wait - for several
 * ranks driven by ONE process, which must enqueue every rank's scan + publish before any rank's wait (kernels of
 * different streams are not guaranteed to run concurrently, so a wait must never sit in front of a peer's publish). */
int carmpc_shard_wait(void* shard, int64_t* d_total_count, void* stream);

/* d_bits: the full bitset (ceil(n_total / 32) words, device memory of this rank) of the last completed step; it stays
 * valid until the second-next sharded call on this window.  h_steps: collective steps done so far.  Synchronous (the
 * step counter lives in device memory: the launch arguments of a collective step never change, so a step can be captured
 * in a CUDA graph and replayed). */
int carmpc_shard_result(void* shard, const uint32_t** d_bits, int64_t* h_steps);
/* Synchronous health check: fails if a peer never published its flag (the exchange kernel gives up after 5 s). */
int carmpc_shard_check(void* shard);

/* ------------------------------------------------------------------------------------------------
 * (B) batched condensed MPC QP
 *
 *   min_u 1/2 u'Hu + (F (x0 - xref))'u
 *   s.t.  lo - Gx x0 - Gc c <= G u <= hi - Gx x0 - Gc c      (m general rows, lo = -inf: one-sided)
 *         lb <= u <= ub                                      (n box rows)
 *         pre_lo <= Px x0 + Pc c <= pre_hi                   (k rows that do not involve u)
 *
 * with x0 (4) the per-sample state, xref (4) the per-batch target (lib/mpc.py:320 / :463) and
 * c (optional, scalar per sample) a constant-disturbance estimate (lib/mpc.py:637).  H, F, G, Gx are
 * lib/matrix_gen.py's H, h and the reference's constraint stacks multiplied into S and T
 * (lib/mpc.py:319-332); see carmpc_b200/condensed.py.
 * ---------------------------------------------------------------------------------------------- */

typedef struct carmpc_qp_opts {
    double rho;            /* ADMM penalty on the scaled problem; <= 0 (default): 320 / n^2 in [0.02, 0.4] */
    double alpha;          /* over-relaxation (default 1.8)                                          */
    double eps_abs;        /* ADMM stop: fixed-point residual, unscaled, abs + rel (default 3e-3;    */
    double eps_rel;        /*   the float64 polish, not this tolerance, sets the final accuracy)     */
    double eps_prim_inf;   /* primal infeasibility certificate tolerance (default 1e-4)              */
    int32_t max_iter;      /* per sample (default 4000)                                              */
    int32_t check_every;   /* residual / certificate test cadence in iterations; <= 0 (default): 14  */
                           /*   for n <= 20 variables, else 10                                       */
    int32_t scaling_iters; /* Ruiz equilibration passes on the host (default 15; 0 = none)           */
    int32_t polish;        /* 1 (default): float64 active-set polish with a KKT check after the      */
                           /*   float32 ADMM; 0: return the raw ADMM iterate                         */
} carmpc_qp_opts;

void carmpc_qp_default_opts(carmpc_qp_opts* opts);

/* Host setup: equilibrate, form K = Hs + rho (Gs'Gs + L^2), invert by Cholesky in float64, analyse the structure
 * (independent chains, causal rows), build the polish matrices, upload.
 * Gc / Pc may be NULL (no disturbance term).  n <= 160; at most 392 general rows with a finite bound; k <= 64. */
int carmpc_qp_create(int n, int m, int k, const double* h_H, const double* h_F, const double* h_G,
                     const double* h_Gx, const double* h_Gc, const double* h_lo, const double* h_hi,
                     const double* h_lb, const double* h_ub, const double* h_Px, const double* h_Pc,
                     const double* h_pre_lo, const double* h_pre_hi, const carmpc_qp_opts* opts,
                     void** handle);

/* Host-only view of the setup (no CUDA call): scaled matrices exactly as they are uploaded.
 * which: 0 D(n) 1 Eg(m) 2 Eb(n) 3 c(1) 4 Kinv(n*n) 5 Gs(m*n) 6 lambda(n)
 *        7 tiling: [samples per lane, stage-A groups per warp, stage-B groups per warp, matrices in shared memory,
 *                   shared bytes, executed flop per sample-iteration, dense flop per sample-iteration, K, padded rows,
 *                   padded variables].
 *        10..26 the padded, permuted float32 device images as float64 (P, Gs, Gs', bounds, tiling tables; see
 *        qp_api.cu) - used by the tests to re-run the kernel's arithmetic on the host.
 *        30..43 the tensor-core form (qp_admm_tc.cu): 30 geometry [has a tensor-core form, padded variables, padded rows,
 *        matrices resident, A stages, B stages, B stage bytes, shared bytes, then per product: image offset, bytes per
 *        chunk pair, chunks, k-steps, MMA N], 31 the chunk images as float32 words, 32..43 the per-row tables.
 * Returns the count (written when h_out != NULL).  A handle created on a machine without a CUDA device keeps this
 * view working; its solve calls return CARMPC_ERR_CUDA. */
int carmpc_qp_get_setup(void* qp, int which, double* h_out, int capacity);

/* Solve `batch` QPs.  d_x0: SoA, 4 arrays of `batch` float64 (x, y, psi, v).  h_xref: 4 host doubles.
 * d_c: nullable per-sample disturbance scalar.
 * Outputs (all device, any may be NULL except d_status):
 *   d_u0        2 x batch float64 SoA: first input of the optimal sequence (what .step returns)
 *   d_objective batch float64: 1/2 u'Hu + q'u at the returned point (the reference's `cost`)
 *   d_status    batch int32 (CARMPC_QP_*)
 *   d_iters     batch int32
 *   d_u_full    batch x n float64, row-major per sample (u_horizon of the reference)
 * d_warm (nullable): batch x (m + n) float32 solver state, read if warm_in != 0, written if warm_out != 0.
 * The call synchronises `stream` (it reads back how many samples need the second, tighter pass). */
int carmpc_qp_solve_batch(void* qp, const double* d_x0, const double* h_xref, const double* d_c,
                          int64_t batch, double* d_u0, double* d_objective, int32_t* d_status,
                          int32_t* d_iters, double* d_u_full, float* d_warm, int warm_in, int warm_out,
                          void* stream);

/* Region-of-attraction maps (the grid search of the reference's paper section III-E: lib/mpc.py:318-338 evaluated
 * on a grid of initial states): neighbouring states mostly share their active set, so only a sub-lattice of
 * "anchor" samples is solved cold (ADMM + polish); every other sample i first tries the certified active set of its
 * anchor d_seed[i] in the float64 polish (one Schur-complement solve + KKT certificate, repaired a few rounds) and
 * runs ADMM iterations only if that does not certify (set too different, or outside the region of attraction).
 * d_seed: batch int32; d_seed[i] == i (or out of range) marks an anchor; a follower's seed must be an anchor.
 * Results are the same certified optima / infeasibility flags as carmpc_qp_solve_batch, whatever the seeds are.
 * h_seeded (nullable): number of samples certified from their seed without any ADMM iteration. */
int carmpc_qp_solve_seeded(void* qp, const double* d_x0, const double* h_xref, const double* d_c,
                           const int32_t* d_seed, int64_t batch, double* d_u0, double* d_objective,
                           int32_t* d_status, int32_t* d_iters, double* d_u_full, int64_t* h_seeded,
                           void* stream);

/* Region-of-attraction map from the host: the states are the C-order tensor grid of four axes (h_axes: the axes
 * concatenated, dims[k] points each, 1..4096; axis k is state component axis_to_state[k]), expanded on the device.
 * block (nullable = every point cold): points per axis of the lattice blocks whose centre points are the anchors
 * of carmpc_qp_solve_seeded.  Outputs as carmpc_qp_solve_host (h_u0 batch x 2 row-major, any may be NULL except
 * h_status); batch = dims[0] dims[1] dims[2] dims[3].  This is the sampled counterpart of the reference's exact
 * but impractical projection lib/in_adm_set.py:4-77 ("grid search" of the paper, section III-E). */
int carmpc_qp_map_host(void* qp, const double* h_axes, const int32_t dims[4], const int32_t axis_to_state[4],
                       const int32_t block[4], const double* h_xref, double* h_u0, double* h_objective,
                       int32_t* h_status, int32_t* h_iters, int64_t* h_seeded);

/* carmpc_qp_solve_batch (d_seed == NULL: cold, no warm state) or carmpc_qp_solve_seeded (d_seed != NULL), with the same
 * results, that also exports the certificate behind every verdict.  d_cert: batch x (m + n + k) float64, row-major per
 * sample, in the row space of the handle: the m general rows, the n box rows and the k u-independent rows exactly as
 * passed to carmpc_qp_create.  Positive means "against the upper bound", negative "against the lower bound".
 *   CARMPC_QP_SOLVED      the multipliers of the float64 KKT certificate: H u + F (x0 - xref) + G' lam_g + lam_b = 0,
 *                         non-zero only on rows the polish certified as active; zero on the k rows.
 *   CARMPC_QP_INFEASIBLE  the Farkas ray y the library checked: G' y_g + y_b = 0 and the support value
 *                         sum_i (y_i+ hi_i(x0, c) - y_i- lo_i(x0, c)) over all m + n + k rows is negative.  A violated
 *                         u-independent row is y = +-1 on that row.  A non-finite state has no certificate (zero row).
 *   CARMPC_QP_MAX_ITER    zeros.
 * Returns CARMPC_ERR_INVALID when the handle has opts.polish == 0 (no certificate without the polish). */
int carmpc_qp_solve_certified(void* qp, const double* d_x0, const double* h_xref, const double* d_c,
                              const int32_t* d_seed, int64_t batch, double* d_u0, double* d_objective,
                              int32_t* d_status, int32_t* d_iters, double* d_u_full, double* d_cert,
                              int64_t* h_seeded, void* stream);

/* Derivatives of certified solutions (carmpc_qp_solve_certified outputs) w.r.t. p = (x, y, psi, v, c): the state and
 * the per-sample disturbance (its column is zero for a handle without Gc).  A solved sample's certificate row names its
 * active rows S; on the critical region of S the optimal u is affine in p (explicit MPC), and
 *   d_jac       batch x rows x 5 float64 (nullable): du_r/dp_k for the leading `rows` variables (1 <= rows <= n; rows = 2
 *               is du0/dp, the local gain of the MPC law)
 *   d_grad_obj  batch x 5 float64 (nullable): dV/dp of the returned objective V
 *   d_flags     batch int32: bit 0 DERIVATIVE  u* is differentiable at p and d_jac is its derivative;
 *               bit 1 WEAK  a row outside S is at a bound (within 1e-8) or a multiplier on S is within the sign tolerance
 *                     (1e-9 (1 + max |lambda|)) of 0: d_jac is the derivative of the affine piece of S, a one-sided
 *                     derivative for perturbations that keep those rows inactive;
 *               bit 2 DEPENDENT  S is linearly dependent: d_jac comes from the independent subset (rows in index order);
 *               bit 3 TOO_MANY_ROWS  more than 64 rows in S (no solver certificate has that many): d_jac is NaN.
 * d_x0: SoA 4 x batch; d_c nullable (the disturbance of the solve); d_status, d_u_full (batch x n) and d_cert
 * (batch x (m + n + k)) as the certified solve returned them.  Samples with status != 0: NaN in d_jac and d_grad_obj,
 * flags 0.  Only enqueues work on `stream`.  CARMPC_ERR_INVALID for a handle with opts.polish == 0. */
int carmpc_qp_sensitivity(void* qp, const double* d_x0, const double* d_c, int64_t batch, const int32_t* d_status,
                          const double* d_u_full, const double* d_cert, int rows, double* d_jac,
                          double* d_grad_obj, int32_t* d_flags, void* stream);

/* Independent float64 checker of certificates for a QP in the general two-sided form
 *     min 1/2 u'Hu + (F (x0 - xref))'u    lo - Gx x0 - Gc c <= G u <= hi - Gx x0 - Gc c ,   lb <= u <= ub
 * with R general rows (a one-sided stack is lo = -inf), stated by the caller: it shares nothing with a QP handle.
 * n <= 160, R <= 16000; Gc may be NULL.  H (n x n), F (n x 4), G (R x n), Gx (R x 4) row-major. */
int carmpc_qp_checker_create(int n, int R, const double* h_H, const double* h_F, const double* h_G,
                             const double* h_Gx, const double* h_Gc, const double* h_lo, const double* h_hi,
                             const double* h_lb, const double* h_ub, void** handle);

/* Checks one certificate row per sample (d_cert: batch x (R + n), general rows then box, sign convention of
 * carmpc_qp_solve_certified) against d_status / d_u_full (batch x n).  d_x0: SoA 4 x batch; d_c nullable.
 * d_resid: batch x 4 float64.  Status 0: [primal violation, stationarity, multiplier against an infinite bound,
 * complementarity], all relative (qp_check.cu states the scales).  Status 1: [support value of the ray with its box part
 * completed as -G'y_g, its rounding scale, |G'y_g + y_b|_inf of the given box part relative to max_j sum_i |G_ij y_i|,
 * mass against infinite bounds]; the ray is a proof iff the last is 0 and support < -4e-12 scale.  Status 2: NaN. */
int carmpc_qp_check(void* checker, const double* d_x0, const double* h_xref, const double* d_c, int64_t batch,
                    const int32_t* d_status, const double* d_u_full, const double* d_cert, double* d_resid,
                    void* stream);

/* Host-buffer convenience: h_x0 is batch x 4 row-major (AoS, as the reference passes states). */
int carmpc_qp_solve_host(void* qp, const double* h_x0, const double* h_xref, const double* h_c, int64_t batch,
                         double* h_u0 /* batch x 2 */, double* h_objective, int32_t* h_status,
                         int32_t* h_iters, double* h_u_full);

/* Sum over the last solve of the per-sample iteration counts and launches issued (for roofline
 * accounting); both int64. */
int carmpc_qp_last_stats(void* qp, int64_t* h_total_iters, int64_t* h_launches);

/* Histogram of the float64 polish over the last solve (20 int64): [r] samples certified after r repair rounds
 * (r = 0..9), [10] handed back to the ADMM, [11] samples whose first round used an anchor's multiplier map,
 * [12] samples certified by that map alone (seeded solve), [13] samples proven infeasible by their anchor's Farkas
 * certificate, [14] max_iter samples proven infeasible by the certificate of their own final ADMM state,
 * [15] samples proven infeasible the same way before the second ADMM pass. */
int carmpc_qp_polish_stats(void* qp, int64_t* h_hist16);

/* Which ADMM kernel large first passes (at least 128 samples per SM) run on.
 *   mode 0  the FFMA tile kernel always;
 *   mode 1  (default) the tcgen05 kernel where it measured faster: problems whose matrices the FFMA kernel cannot keep in
 *           shared memory (horizon 40 of the shipped environments);
 *   mode 2  the tcgen05 kernel whenever the problem has a tensor-core form: up to 256 general rows and
 *           2 rows + variables <= 512 columns of tensor memory (horizons up to 40), or - larger problems - the same for
 *           every independent chain of the variable graph (horizon 80 of RoadEnv / RoadOneCarEnv: the acceleration and
 *           steering chains are solved as two passes of the kernel and their verdicts merged);
 *   mode 3  mode 2 with cycle counters (a measuring aid: where the roles of the kernel wait);   mode < 0 only queries.
 * The tcgen05 kernel: 128-sample tiles as the M dimension of kind::tf32 MMAs, 3xTF32 split, state and accumulators in
 * tensor memory.  Both kernels run the same iteration; the float64 polish certifies the results of either.
 * h_info (nullable, 16 int64): [0] mode, [1] number of tensor-core parts (0: no tensor-core form, 1: the whole problem,
 * > 1: one pass per independent chain), [2] samples the tcgen05 kernel
 * took in the last solve, [3] 1 if its matrices stay resident in shared memory (0: streamed from L2 every iteration),
 * [4..13] mode 3: cycles summed over the CTAs of the last tcgen05 launch - MMA thread: round total, waiting for A
 * chunks, waiting for B chunks; compute thread 0: waiting for x~, waiting for z^, waiting for a free A stage, retire /
 * refill, round total, rounds; B stream thread: waiting for a free stage; [14], [15] compute thread 0: cycles in the
 * generic-to-async proxy fence of its A-chunk writes, and in fence + warp synchronisation. */
int carmpc_qp_tensor_mode(void* qp, int mode, int64_t* h_info);

/* ------------------------------------------------------------------------------------------------
 * Monte-Carlo closed loop against the nonlinear bicycle (lib/simulator.py:51-69), in the order of
 * examples/run_MPCOutputFB.py:29-41: plant step with the previous input (first [0,0]), observer
 * update (mode 1, lib/mpc.py:448) or direct state (mode 0), QP, repeat.
 *   h_A (4x4), h_B (4x2), h_C (3x4), h_L (4x3) row-major; dt, l1 as in the reference (0.2, 3.5).
 *   d_x_init, d_xhat_init: SoA 4 x runs.  d_final: SoA 4 x runs.  d_fail_step: int32, -1 = none.
 *   d_traj (nullable): steps x 4 x runs float64.  d_u_log (nullable): steps x 2 x runs.
 * A run whose QP is infeasible at step t stops there (the reference raises) and keeps its state.
 * warm_start: 0 = every QP cold; 1 = the previous step's certified active set / ADMM state is reused and the steps are
 * only enqueued (every sample count stays on the device, no host synchronisation inside the loop); 2 = the same reuse
 * with host-sized launches (three count read-backs per step: the round-1 form, kept to time one against the other). */
int carmpc_closed_loop(void* qp, int mode, const double* h_A, const double* h_B, const double* h_C,
                       const double* h_L, const double* h_xref, double dt, double l1, int steps, int warm_start,
                       const double* d_x_init, const double* d_xhat_init, int64_t runs, double* d_final,
                       int32_t* d_fail_step, double* d_traj, double* d_u_log, int64_t* h_total_iters,
                       void* stream);

/* Closed loops of the disturbance-estimating output-feedback controller (MPCOutputFBWithDisturbance, lib/mpc.py:329-396):
 * the same loop, with a constant scalar disturbance per run and an augmented observer.  Step k of a run:
 *   s  = s + dt * f(s, u_prev);   s = s + Bd_plant * d_r          (plant: Euler step, then the true disturbance)
 *   y  = C s + Cd_plant * d_r
 *   i  = y - C x^ - Cd d^;   x^' = A x^ + Bd d^ + B u_prev + L1 i;   d^' = d^ + L2 . i
 *   QP at x0 = x^', c = d^' (bounds shifted by Gc c), x_ref = h_xref
 * The QP handle's Gc must describe the same Bd (BatchQP.from_controller of a controller with that Bd); a handle whose Gc
 * is zero is allowed (c then has no effect).  Infeasible or undecided QPs stop the run (d_fail_step), as in
 * carmpc_closed_loop; "infeasible" verdicts carry a float64 certificate of the disturbance-shifted problem.
 * Non-finite gains are rejected; a non-finite d^ or state of one run makes that run's QP infeasible.
 *   dm: model and gains (L1 4x3 row-major).  d_x_init, d_xhat_init (nullable: x_init): SoA 4 x runs.
 *   d_dhat_init (nullable: 0), d_d_plant (nullable: 0, the per-run d_r), d_dhat_final (nullable): runs float64.
 *   d_traj, d_u_log as in carmpc_closed_loop; d_dhat_log (nullable): steps x runs, d^ the QP of each step used.
 * warm_start 0 / 1 / 2 as in carmpc_closed_loop. */
typedef struct carmpc_disturbance_model {
    double Bd[4], Cd[3], L1[12], L2[3];   /* controller: disturbance model and observer gains (L1 4x3 row-major) */
    double Bd_plant[4], Cd_plant[3];      /* how the true per-run disturbance enters the plant state / output    */
} carmpc_disturbance_model;

int carmpc_closed_loop_disturbance(void* qp, const double* h_A, const double* h_B, const double* h_C,
                                   const carmpc_disturbance_model* dm, const double* h_xref, double dt, double l1,
                                   int steps, int warm_start, const double* d_x_init, const double* d_xhat_init,
                                   const double* d_dhat_init, const double* d_d_plant, int64_t runs, double* d_final,
                                   double* d_dhat_final, int32_t* d_fail_step, double* d_traj, double* d_u_log,
                                   double* d_dhat_log, int64_t* h_total_iters, void* stream);

/* Closed loops with random process and measurement noise, and a monitor of the true plant state (modes 0, 1, 2 of the two
 * functions above).  Step k of a run still running at the start of step k:
 *   s = s + dt * f(s, u_prev);   mode 2: s = s + Bd_plant * d_r;   s = s + Lw z_w      (process noise)
 *   s is stored to d_final / d_traj, then checked against the monitor rows [a | b]: fma(a3, v, fma(a2, psi, fma(a1, y,
 *   a0 * x))) <= b for every row (the chain of carmpc_membership_bitset mode 0; a non-finite state violates)
 *   v = Lv z_v;   mode 0: the QP sees s + v[0..3];  mode 1: y = C s + v[0..2];  mode 2: y = C s + Cd_plant d_r + v[0..2]
 *   observer and QP as in carmpc_closed_loop / carmpc_closed_loop_disturbance.
 * z_w, z_v: four standard normals each.  Philox4x64-10 with key (seed, 0) at counter (first_run + run, k, j, 0), j = 0
 * for z_w and 1 for z_v, gives words x0..x3; (x0, x1) and (x2, x3) each give two normals by Box-Muller:
 *   ua = ((x0 >> 11) + 1) 2^-53,  ub = (x1 >> 11) 2^-53,  z0 = sqrt(-2 ln ua) cos(2 pi ub),  z1 = ... sin(2 pi ub).
 * The draws depend only on (seed, first_run + run, k, j): not on the batch, warm_start or which runs still run, so a run
 * set split over calls (first_run = the offset of each part) draws what one call would.
 * A violation never stops a run.  d_violation_step / d_violation_row (runs int32, -1 none): the first step with a
 * violation and the lowest violated row (caller's order) at that step.  d_violations_per_step (steps int32): runs
 * violating at step k.  Stopped runs are neither moved nor counted; a run whose QP fails at step k was moved and checked
 * at step k.
 *   mode 0: h_C, h_L ignored;  mode 1: h_C, h_L (as carmpc_closed_loop);  mode 2: h_C and dm (h_L ignored).
 *   d_dhat_init, d_d_plant, d_dhat_final, d_dhat_log: mode 2 only (as carmpc_closed_loop_disturbance).
 *   noise (nullable: no noise).  h_monitor_Ab (nullable: no monitor): host rows x 5, 1 <= monitor_rows <= 512, finite;
 *   the monitor outputs are nullable and need rows.
 * With noise = NULL and no monitor the results are those of carmpc_closed_loop / carmpc_closed_loop_disturbance.
 * CARMPC_ERR_INVALID for non-finite factors or gains, first_run < 0, bad monitor rows, monitor outputs without rows, mode
 * 2 without dm; CARMPC_ERR_CUDA on a handle created without a device. */
typedef struct carmpc_loop_noise {
    uint64_t seed;
    int64_t first_run;      /* global id of run 0 of this call */
    double Lw[16];          /* process-noise factor, 4 x 4 row-major: w = Lw z_w   */
    double Lv[16];          /* measurement-noise factor, 4 x 4 row-major: v = Lv z_v */
} carmpc_loop_noise;

int carmpc_closed_loop_stochastic(void* qp, int mode, const double* h_A, const double* h_B, const double* h_C,
                                  const double* h_L, const carmpc_disturbance_model* dm, const double* h_xref, double dt,
                                  double l1, int steps, int warm_start, const double* d_x_init, const double* d_xhat_init,
                                  const double* d_dhat_init, const double* d_d_plant, int64_t runs, double* d_final,
                                  double* d_dhat_final, int32_t* d_fail_step, double* d_traj, double* d_u_log,
                                  double* d_dhat_log, const carmpc_loop_noise* noise, const double* h_monitor_Ab,
                                  int monitor_rows, int32_t* d_violation_step, int32_t* d_violation_row,
                                  int32_t* d_violations_per_step, int64_t* h_total_iters, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Device micro-benchmarks used as roofline denominators that MEASURED_PEAKS.json does not carry.
 * which: 0 = FP32 FFMA TFLOP/s (uniform multiplier), 1 = FP64 DFMA TFLOP/s, 2 = HBM copy GB/s (read+write),
 *        3 = FP32 TFLOP/s of a shared-memory-fed 8x8 register-tile product (the practical ceiling of a tile loop). */
int carmpc_measure_peak(int which, double* h_value);

#ifdef __cplusplus
}
#endif
#endif /* CARMPC_H */
