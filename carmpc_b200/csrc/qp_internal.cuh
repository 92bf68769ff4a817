// Internal layout of the batched condensed-QP solver (shared by qp_setup.cu, qp_admm.cu, qp_polish.cu, qp_api.cu and
// closed_loop.cu).  Nothing here is part of the C ABI.
//
// Problem (include/carmpc.h):   min 1/2 u'Hu + (F (x0 - xref))'u
//                               lo - Gx x0 - Gc c <= G u <= hi - Gx x0 - Gc c ,   lb <= u <= ub
// One instance per initial state x0; H, F, G, Gx and the bounds are shared by the whole batch, which is what
// makes the ADMM linear operator one dense matrix applied to a (variables x samples) tile.
//
// Device algorithm (two kernels per pass):
//   1. admm_kernel   float32 OSQP-style ADMM on the Ruiz-equilibrated problem, in the single-vector form
//                        c = clip(w) ; x~ = P (2c - w) + x~0 ; z = A_s x~ ; w += alpha (z - c)
//                    with P = rho K^-1 A_s' precomputed on the host (K = H_s + rho A_s'A_s is shared).  It only has
//                    to identify the active set / prove infeasibility.
//   2. polish_kernel float64 active-set solve through the Schur complement  (A_act H^-1 A_act') lambda = ... with
//                    the shared H^-1, A H^-1, A H^-1 A' precomputed; verifies primal feasibility and multiplier
//                    signs (a KKT certificate), repairs the set a few times, and produces u to ~1e-10.
#pragma once

#include <atomic>
#include <vector>

#include "common.cuh"

namespace carmpc {

constexpr int kRA = 5;            // rows of x~ per thread tile in stage A
constexpr int kRB = 7;            // constraint rows per thread tile in stage B
constexpr int kAdmmWarps = 8;
constexpr int kAdmmThreads = kAdmmWarps * 32;
constexpr int kMaxN = 160;        // variables (2 x horizon 80)
constexpr int kMaxM = 392;        // general rows (8 warps x 7 groups x 7 rows)
constexpr int kPolishMaxActive = 64;
// KKT tolerances of the polish's certificate (qp_polish.cu), shared with the sensitivity pass (qp_sensitivity.cu) so that
// "a row at its bound" and "a multiplier of the right sign" mean what the certificate can distinguish:
constexpr double kFeasTol = 1e-8;     // a row is satisfied when it exceeds its bound by at most this (absolute)
constexpr double kSignTol = 1e-9;     // a multiplier is wrong-signed below -kSignTol (1 + max |lambda|)
constexpr int kPolishStats = 20;       // counters of carmpc_qp_polish_stats
constexpr int kFirstPassIters = 100;  // iteration cap of the first ADMM pass (stragglers continue in the second pass)

enum SlotState : int { kSlotIdle = -1, kSlotRunning = 0, kSlotSolved = 1, kSlotInfeasible = 2, kSlotMaxIter = 3,
                       kSlotPreInfeasible = 4 };

// status codes between the kernels (the ABI codes are CARMPC_QP_*)
constexpr int kStatusNeedsMoreAdmm = 3;      // polish could not certify: re-run ADMM tighter

struct AdmmTables {
    // matrices (float32)
    const float* P;        // [nA_rows][ktot]      rho K^-1 [Gs' | diag(lam)], columns in V order
    const float* Gs;       // [m_phys][npad4]      scaled general rows, physical (owner) order, permuted variables
    const float* GsT;      // [nA_rows][mv4]       Gs', columns in V order (certificate pass)
    // per physical general row
    const double* his;     // [m_phys]   Eg * hi        (pad rows: 3e38)
    const double* Gxs;     // [m_phys][4]
    const double* Gcs;     // [m_phys]
    const float* width;    // [m_phys]   Eg * (hi - lo), +inf for one-sided and pad rows
    const float* Einv_g;   // [m_phys]   1 / Eg         (pad rows: 0)
    const float* Esc_g;    // [m_phys]   Eg             (pad rows: 0)
    const int* vpos;       // [m_phys]   row of V this constraint row writes
    const int* row_id;     // [m_phys]   logical row index, -1 for pad rows
    // per permuted variable
    const float* lam;      // [nA_rows]  Eb * D (scaled box row), 0 for pad
    const float* lbs;      // [nA_rows]
    const float* ubs;      // [nA_rows]
    const float* Einv_b;   // [nA_rows]
    const float* Esc_b;    // [nA_rows]  Eb
    const float* Dinv;     // [nA_rows]
    const float* Dsc;      // [nA_rows]  D (u = D x~)
    const double* KF;      // [nA_rows][4]   x~0 = KF (x0 - xref)
    const int* var_id;     // [nA_rows]  logical variable index, -1 for pad
    // per group of rows
    const int4* segA;      // [nA_rows / kRA]   V ranges (general beg, end, box beg, end), multiples of 4
    const int2* segB;      // [m_phys / kRB]    x~ range (beg, end), multiples of 4
    // rows that do not depend on u: pre_lo <= Px x0 + Pc c <= pre_hi
    const double* Px;
    const double* Pc;
    const double* pre_lo;
    const double* pre_hi;
    int kpre;
    int n, m, mt;                          // logical sizes, mt = m + n
    int nA_rows, m_phys, npad4, mv4, ktot; // padded sizes
    int nGA, nGB;                          // number of row groups in stage A / B
    float rho, alpha, eps_abs, eps_rel, eps_inf;
    int check_every;
};

struct AdmmBatch {
    const double* x0;        // SoA: x0[c * stride + sample]
    int64_t stride;
    const double* cdist;     // nullable, per sample
    double xref[4];
    const int* idx_list;     // nullable: sample = idx_list[q]
    int count;               // number of queue entries
    const int* count_dev;    // nullable: the number of entries lives on the device (count is then an upper bound)
    int narrow;              // host side: always run the narrowest tile (device-sized batches of unknown, usually small, size)
    int* next;               // global work counter (zeroed before launch)
    int8_t* sign;            // [batch][mt]   +1 upper active, -1 lower active
    float* u_admm;           // [batch][n]    unscaled iterate (fallback when the polish cannot certify)
    int* status;
    int* iters;
    float* warm;             // nullable, [batch][mt] scaled w
    int warm_in, warm_out;
    unsigned long long* total_iters;
    float eps_scale;
    int max_iter;
    int iters_accumulate;    // second pass: add to the iteration count of the first
    int write_u;             // also write the ADMM iterate (needed when the polish may pass it through)
    int combine;             // tensor-core kernel, second and later chains of a split problem: merge status / iterations
                             // with what the earlier chains wrote (infeasible if any chain is, solved if all are)
    unsigned long long* prof; // nullable (tensor-core kernel, tensor mode 2): cycle counters summed over the CTAs
};

// Tensor-core form of the ADMM (qp_admm_tc.cu): a tile of 128 samples is the M dimension of tcgen05.mma kind::tf32, the
// shared matrices are the B operands (K-major, 128-byte swizzle, split into a TF32 "hi" image and a TF32 "lo" residual
// image for the 3xTF32 products), the ADMM state of the general rows and the accumulators live in tensor memory.
// Everything is in logical order (live general rows, then variables); pads are inert (zero matrix rows / columns).
//   product 0   x~ (np)   = [V_b (np) | e (16) | V^_g (mp)] . B0'      K0 = np + 16 + mp
//   product 1   z^ (mp)   = [x~  (np) | e (16)] . B1'                  K1 = np + 16
//   product 2   Gs'dy (np) = [dy (mp)] . B2'                           K2 = mp          (certificate, checked iterations)
// e = per-sample constants as exact TF32 pieces: x0_c as hi / mid / lo (c = 0..3), 1, the disturbance c as hi / mid / lo.
// General rows are kept shifted by their per-sample upper bound h = his - Gxs x0 - Gcs c (w^ = w - h, z^ = z - h), which
// makes their clip bounds (-width, 0) sample-independent; the shift enters both products through the e columns.
struct TcTables {
    const unsigned char* img;   // chunk images: chunk k of product p at img + off[p] + k * pair_bytes[p] (hi image, then lo)
    int off[3], pair_bytes[3], nchunks[3], ksteps[3], ncols[3];
    const float* nwd;           // [mp]   -width (scaled; -inf: one-sided or pad row)
    const float* einv_g;        // [mp]   1 / Eg (pads 0)
    const float* hisf;          // [mp]   float copies of his, Gxs, Gcs for the residual norms / support sums (pads 0)
    const float* gxsf;          // [mp][4]
    const float* gcsf;          // [mp]
    const double* his;          // [mp]   (pads 0)
    const double* gxs;          // [mp][4]
    const double* gcs;          // [mp]
    const int* row_id;          // [mp]   logical row, -1 pad
    const float* lam;           // [np]   Eb D (pads 0)
    const float* lb;            // [np]   scaled box (pads -inf / +inf)
    const float* ub;
    const float* einv_b;        // [np]
    const float* nrl;           // [np]   -1 / lam (pads 0)
    const double* kfv;          // [np][4]  x~0 = kfv (x0 - xref)
    const int* var_id;          // [np]   logical variable, -1 pad
    int n, m, mt, np, mp;
    int resident;               // products 0 and 1 stay in shared memory (loaded once); product 2 always streams
    int merged;                 // B_hi and B_lo are consumed as ONE operand of 2 N rows (A_hi fetched once per k-step: two
                                // MMAs instead of three); needs 2 N accumulator columns per product: 3 mp + 2 np <= 512
    int na_stages, nb_stages, b_stage_bytes, resident_bytes;
    int smem_bytes;
    int ok;                     // 0: this problem has no tensor-core form (too large for tensor memory / shared memory)
};

// host images of one part of the tensor-core form (the whole problem, or one independent chain of it)
struct TcPart {
    TcTables t;
    std::vector<unsigned char> img;
    std::vector<float> nwd, einv_g, hisf, gxsf, gcsf, lam, lb, ub, einv_b, nrl;
    std::vector<double> his, gxs, gcs, kfv;
    std::vector<int> row_id, var_id;
};

struct PolishTables {
    const double* H;         // [n][n]
    const double* Hinv;      // [n][n]
    const double* F;         // [n][4]
    const double* Uu;        // [n][4]      u_unc = Uu (x0 - xref),  Uu = -H^-1 F
    const double* AUu;       // [mt][4]     [G; I] Uu
    const double* AH;        // [mt][n]     [G; I] H^-1
    const double* AHA;       // [mt][mt]    [G; I] H^-1 [G; I]'
    const double* Gx;        // [m][4]
    const double* Gc;        // [m]
    const double* hi;        // [mt]  (general rows then box)
    const double* lo;        // [mt]
    const double* G;         // [m][n]      general rows (rows bounded only from below negated, as hi / lo)
    const double* Eg;        // [m]         row scaling of the ADMM (its dual iterate is in scaled units)
    const double* rsign;     // [m]         -1 for a row the setup negated (bounded only from below), else +1
    int n, m, mt;
    int kpre;                // u-independent rows: a certificate row has mt + kpre entries
};

struct PolishBatch {
    const double* x0;
    int64_t stride;
    const double* cdist;
    double xref[4];
    const int* idx_list;
    int count;
    const int* count_dev;    // nullable: the number of list entries lives on the device (count is then an upper bound)
    const int8_t* sign;
    const float* u_admm;
    int* status;             // in: 0 / 2 from ADMM -> out: 0 solved (polished or accepted), 3 needs more ADMM
    double* u0;              // SoA 2 x stride (nullable)
    double* objective;       // nullable
    double* u_full;          // [batch][n] nullable
    int8_t* polished;        // nullable
    int* n_failed;           // device counter of samples set to kStatusNeedsMoreAdmm
    int* failed_list;        // their indices
    int final_pass;          // 1: accept the ADMM iterate when the polish cannot certify
    int rounds;              // repair rounds (-1: default; 0: no polish, pass the ADMM iterate through)
    int na_cap;              // active rows this launch has shared memory for
    int* overflow_list;      // samples with more (nullable: they count as not certified)
    int* n_overflow;
    // active-set reuse (closed loop: the previous step's certified set is tried before any ADMM iteration)
    int precheck;            // 1: also evaluate the u-independent rows / finiteness the ADMM slot refill checks
    const double* Px;        // [kpre][4]
    const double* Pc;        // [kpre]
    const double* pre_lo;
    const double* pre_hi;
    int kpre;
    int8_t* sign_out;        // nullable: the certified active set is written back ([batch][mt])
    int* iters_out;          // nullable: certified samples get 0 iterations
    // active-set seeding (region-of-attraction maps: neighbouring states mostly share their active set)
    const int* seed;         // nullable: sample i starts from the certified set of sample seed[i] (an anchor solved before)
    // multiplier maps of the anchors' critical regions: lambda(x0) = Lam [x0; 1] on the anchor's active rows
    const int* rec_of;       // [batch] record of a sample (-1: none)
    double* rec_lam;         // [records][32][5]
    int* rec_act;            // [records][33]   na (-1: no map), then the active rows in the order of Lam's rows
    int rec_write, rec_read;
    double* cert;            // nullable [batch][mt + kpre]: multipliers of certified samples (carmpc_qp_solve_certified)
    unsigned long long* stats;   // nullable [20]: [r] samples certified after r repair rounds (r = 0..9), [10] not certified,
                                 // [11] round 0 taken from a multiplier map, [12] certified by a multiplier map alone,
                                 // [13] proven infeasible by the anchor's Farkas certificate (or the u-independent rows),
                                 // [14] max_iter samples proven infeasible by the certificate of their own ADMM state,
                                 // [15] samples proven infeasible the same way before the second pass
                                 // [16] samples the final polish could not certify (handed to the float64 fallback),
                                 // [17] of those solved + certified, [18] proven infeasible, [19] left undecided (status 2)
};

// float64 images of the equilibrated problem for the fallback solver (qp_exact.cu), logical order
struct ExactTables {
    const double* Gs;        // [m][n]   Eg G D (rows without a finite bound: zero)
    const double* GsT;       // [n][m]
    const double* Kinv;      // [n][n]   (Hs + rho (Gs'Gs + lam^2))^-1
    const double* lam;       // [n]      Eb D
    const double* Eb;        // [n]
    const double* D;         // [n]
    const double* rowmin;    // [m]      min over the input box of G_i u  (-inf when a needed box side is infinite)
    const double* rowmax;    // [m]      max over the input box of G_i u
    const double* rowabs;    // [m]      sum_j |G_ij| max(|lb_j|, |ub_j|): rounding scale of the two
    double cs, rho, alpha;
};

// Host-side setup product (qp_setup.cu)
struct QPHost {
    int n = 0, m = 0, kpre = 0;
    carmpc_qp_opts opts;
    // scaling (logical order)
    std::vector<double> D, Eg, Eb, Kinv, Gs64;
    double cscale = 1.0;
    // padded device images
    AdmmTables geo;          // sizes only (pointers filled by the handle)
    std::vector<float> P, Gs, GsT, width, Einv_g, Esc_g, lam, lbs, ubs, Einv_b, Esc_b, Dinv, Dsc;
    std::vector<double> his, Gxs, Gcs, KF, Px, Pc, pre_lo, pre_hi;
    std::vector<int> vpos, row_id, var_id;
    std::vector<int4> segA;
    std::vector<int2> segB;
    // polish (logical order, unscaled)
    std::vector<double> H, Hinv, F, G, Uu, AUu, AH, AHA, Gx, Gc, hi, lo;
    std::vector<double> rsign;       // [m] -1 where a row bounded only from below was negated
    // tensor-core form: one part for the whole problem, or one per independent chain (sizes in t; pointers filled by the handle)
    TcTables tc;                     // = tc_parts[0].t
    std::vector<TcPart> tc_parts;
    int ga_per_warp = 0, gb_per_warp = 0, samples_per_lane = 0;
    bool mats_in_smem = false;
    size_t smem_bytes = 0;
    double flops_per_iter = 0;      // executed FFMA * 2 per sample-iteration (structure-aware)
    double flops_per_iter_dense = 0;
};

int qp_host_setup(int n, int m, int k, const double* H, const double* F, const double* G, const double* Gx,
                  const double* Gc, const double* lo, const double* hi, const double* lb, const double* ub,
                  const double* Px, const double* Pc, const double* pre_lo, const double* pre_hi,
                  const carmpc_qp_opts& opts, QPHost* out);

// What one solve is asked to do (host only).  QPHandle::solve / solve_enqueue / solve_seeded take it whole, so that no
// option of a call is left on the handle for the next one.  Device pointers; outputs are nullable except status.
struct SolveRequest {
    const double* x0 = nullptr; int64_t stride = 0;   // SoA x0[c * stride + sample]; every per-sample array has stride
    const double* xref = nullptr;    // host, 4 values
    const double* c = nullptr;       // nullable per-sample disturbance: every stage shifts its bounds by Gc c
    const int* idx = nullptr; int64_t count = 0;       // the samples solved now: idx[0 .. count) (null idx: 0 .. count)
    const int* count_dev = nullptr;  // solve_enqueue: the number of listed samples lives here (count is an upper bound)
    double *u0 = nullptr, *objective = nullptr, *u_full = nullptr;
    int32_t *status = nullptr, *iters = nullptr;
    double* cert = nullptr;          // [stride][mt + kpre] certificate rows, zeroed by the caller
    float* warm = nullptr;           // ADMM state [stride][mt] (null: the workspace's)
    int warm_in = 0, warm_out = 0;
    int reuse = 0;                   // try the certified active set kept in the workspace first
    const int* seed = nullptr;       // with reuse: sample i starts from the certified set of sample seed[i]
    int keep_sign = 0;               // write certified active sets back to the workspace
    int records = 0;                 // seeded solve: anchors export multiplier maps, followers read them
    int hold_stats = 0;              // keep counting into the polish histogram instead of zeroing it
    int keep_total = 0;              // closed loop: the iteration total accumulates on the device, read once at the end
    int certify_shifted = 0;         // run the filter / decide certificates with a disturbance too (the public entry
                                     // points keep max_iter there)
};

// What a solve did (also published as last_total_iters / last_launches for carmpc_qp_last_stats): ADMM iterations (0
// with keep_total), kernel launches, samples certified from the reused active set
struct SolveCounts { int64_t iters = 0, launches = 0, reused = 0; };

// Counters of the solve pipeline (QPHandle::ws_counters, 16 ints).  The indices are fixed: solve() zeroes [0, 8) per call,
// solve_enqueue() [0, 16), solve_seeded() the split pair [8, 10).
constexpr int kCntNext = 0;          // ADMM work counter, first pass
constexpr int kCntFailed = 1;        // first-pass samples the polish could not certify (list ws_failed)
constexpr int kCntNext2 = 2;         // ADMM work counter, second pass
constexpr int kCntFinal = 3;         // n_failed of the final polish (a final pass lists nothing)
constexpr int kCntOverflow = 4;      // polish samples over the small active-set budget (list ws_overflow)
constexpr int kCntReuseFailed = 5;   // samples the reused active set did not certify (list ws_failed0)
constexpr int kCntRest = 6;          // samples the empty active set did not settle (list ws_rest)
constexpr int kCntSurvivors = 7;     // samples the Farkas filter did not prove infeasible (list ws_overflow)
constexpr int kCntAnchors = 8;       // seeded split: anchors (list ws_anchor), then followers (list ws_follow) at 9
constexpr int kCntUnproven = 11;     // samples the second pass left without a proof (list ws_unproven)
constexpr int kCntExactFinal = 12;   // n_failed of the fallback's polish (a final pass lists nothing)
constexpr int kCntVerify2 = 13;      // second-pass "infeasible" verdicts without a certificate (list ws_overflow)
constexpr int kCounters = 16;
// ws_overflow holds three lists in turn: the polish's overflow (kCntOverflow, refilled by every polish launch), the Farkas
// filter's survivors (kCntSurvivors, copied to ws_failed at once) and the second verify's failures (kCntVerify2, never
// read back: the exact fallback finds them by their status).

struct QPHandle;
struct QPBusyGuard {
    std::atomic<bool>* flag;
    bool acquired;
    explicit QPBusyGuard(std::atomic<bool>& f) : flag(&f) { bool expect = false; acquired = f.compare_exchange_strong(expect, true); }
    ~QPBusyGuard() { if (acquired) flag->store(false); }
};
int admm_launch(QPHandle* q, const AdmmBatch& b, cudaStream_t st);
// tcgen05 form of the same iteration (qp_admm_tc.cu); admm_launch picks it for large first passes
int admm_tc_launch(QPHandle* q, const AdmmBatch& b, cudaStream_t st);
bool admm_tc_usable(const QPHandle* q, const AdmmBatch& b);
int polish_launch(QPHandle* q, const PolishBatch& b, cudaStream_t st);
// the empty active set tried first (one thread per sample); samples it does not settle are appended to d_rest
int polish_unconstrained_launch(QPHandle* q, const PolishBatch& b, int* d_rest, int* d_n_rest, cudaStream_t st);
// The certificate launches take the per-sample arrays (x0, c, status, outputs), the histogram and the certificate rows
// from the call's polish batch `b`, and work on the samples d_list[0 .. count) (d_count: the count lives on the device).
// infeasible anchors of a seeded map: turn the ADMM dual iterate into an exact Farkas certificate, affine in x0
int farkas_export_launch(QPHandle* q, const PolishBatch& b, const int* d_list, int count, const float* d_warm, cudaStream_t st);
// before the second pass: samples the certificate of their first-pass state proves infeasible are done, the rest is listed
int farkas_filter_launch(QPHandle* q, const PolishBatch& b, const int* d_list, int count, const float* d_warm,
                         int* d_survivors, int* d_n_survivors, cudaStream_t st);
// samples that ran out of ADMM iterations: a valid certificate from their final ADMM state makes them proven infeasible
int farkas_decide_launch(QPHandle* q, const PolishBatch& b, const int* d_list, int count, const int* d_count,
                         const float* d_warm, cudaStream_t st);
// ADMM verdicts "infeasible" are only accepted with a float64 certificate: the others re-enter the second pass
int farkas_verify_launch(QPHandle* q, const PolishBatch& b, const int* d_list, int count, const int* d_count,
                         const float* d_warm, int* d_failed, int* d_n_failed, cudaStream_t st);
// float64 fallback for what the second pass could not prove (qp_exact.cu); *h_handled: the number of samples it took
int exact_fallback(QPHandle* q, const PolishBatch& b, const int* d_list, int count, const int* d_count, float* d_warm,
                   int* d_iters, cudaStream_t st, int* h_handled);
size_t admm_smem_bytes(const QPHost& h, int samples_per_lane, bool mats_in_smem);
// derivatives of certified solutions (qp_sensitivity.cu); d_x0 SoA with stride = batch, d_jac / d_grad nullable
int sensitivity_launch(QPHandle* q, const double* d_x0, const double* d_c, int64_t batch, const int32_t* d_status,
                       const double* d_u_full, const double* d_cert, int rows, double* d_jac, double* d_grad,
                       int32_t* d_flags, cudaStream_t st);

// Certificate rows (carmpc_qp_solve_certified) are in the caller's orientation: entry i of a general row the setup negated
// changes sign, so that positive always means "against the upper bound" of the row as passed to carmpc_qp_create.
// A violated u-independent row is an infeasibility proof by itself: y = +1 (above pre_hi) or -1 (below pre_lo) on the
// first such row, zeros elsewhere (its G part is zero).  A non-finite state has no certificate: the row stays zero.
// The whole warp writes the row.
__device__ __forceinline__ void store_pre_certificate(double* row, int mt, int kpre, const double* Px, const double* Pc,
                                                      const double* pre_lo, const double* pre_hi, const double (&x0)[4],
                                                      double cd, int lane) {
    for (int e = lane; e < mt + kpre; e += 32) row[e] = 0.0;
    __syncwarp();
    if (lane != 0) return;
    for (int k = 0; k < kpre; ++k) {
        const double v = Px[k * 4 + 0] * x0[0] + Px[k * 4 + 1] * x0[1] + Px[k * 4 + 2] * x0[2] + Px[k * 4 + 3] * x0[3] + Pc[k] * cd;
        if (v > pre_hi[k]) { row[mt + k] = 1.0; return; }
        if (v < pre_lo[k]) { row[mt + k] = -1.0; return; }
    }
}

struct QPHandle : HandleBase {
    QPHost host;
    AdmmTables admm;
    TcTables tc;                                 // = tc_parts[0]
    std::vector<TcTables> tc_parts;              // device tables of every part (one, or one per independent chain)
    int tensor_mode = 1;                         // 0: FFMA kernel only; 1: tcgen05 kernel where it is faster; 2: wherever possible; 3: 2 + cycle counters
    int64_t last_tc_samples = 0;                 // samples the tcgen05 kernel took in the last solve
    unsigned long long* ws_prof = nullptr;       // [16] cycle counters of the tcgen05 kernel (tensor mode 2)
    PolishTables polish;
    ExactTables exact;
    std::vector<void*> allocations;
    // per-batch workspace (grown on demand)
    int64_t ws_batch = 0;
    int8_t* ws_sign = nullptr;
    float* ws_u = nullptr;
    int* ws_status = nullptr;
    int* ws_iters = nullptr;
    int* ws_failed = nullptr;
    int* ws_failed0 = nullptr;                   // samples whose reused active set did not certify
    int* ws_rest = nullptr;                      // samples the empty active set does not settle
    int* ws_anchor = nullptr;                    // seeded solve: samples solved cold (anchors) / from a seed (followers)
    int* ws_follow = nullptr;
    int* ws_rec_of = nullptr;                    // [batch] record index of an anchor
    double* ws_rec_lam = nullptr;                // multiplier maps of the anchors (grown on demand, capped)
    int* ws_rec_act = nullptr;
    int64_t rec_cap = 0;
    unsigned long long* ws_polish_stats = nullptr;   // [kPolishStats] histogram of the polish launches of the last solve
    int* ws_overflow = nullptr;
    int* ws_unproven = nullptr;                  // samples the second pass left without a proof (float64 fallback)
    int* ws_counters = nullptr;                  // [kCounters], indices kCnt*
    unsigned long long* ws_total_iters = nullptr;
    int8_t* ws_polished = nullptr;
    float* ws_warm = nullptr;                    // ADMM state of every sample (warm start of the second pass)
    // device side of the host-buffer entry point (grown on demand, kept across calls)
    int64_t io_cap = 0, io_full_cap = 0;
    double *io_x0_aos = nullptr, *io_x0 = nullptr, *io_c = nullptr, *io_u0 = nullptr, *io_u0_aos = nullptr, *io_obj = nullptr,
           *io_full = nullptr;
    int32_t *io_status = nullptr, *io_iters = nullptr, *io_seed = nullptr;
    double* io_axes = nullptr;                   // grid axes of carmpc_qp_map_host
    int ensure_io(int64_t batch, bool want_full);
    int64_t last_total_iters = 0, last_launches = 0;   // carmpc_qp_last_stats: the counts of the last (seeded) solve
    int sm = 148;
    bool host_only = false;
    // per-call state lives in the handle (workspace, counters): one call at a time.  A second call entering while one is
    // in flight (another host thread) is refused instead of corrupting both.
    std::atomic<bool> busy{false};
    ~QPHandle() override;
    int ensure_workspace(int64_t batch);
    // full solve on device buffers; counts (nullable) receives what the call did
    int solve(const SolveRequest& r, cudaStream_t st, SolveCounts* counts = nullptr);
    // The same pipeline for a warm-started sequence (closed loop), with every sample count left on the device: the list
    // r.idx holds *r.count_dev <= r.count entries, the previous step's certified active sets are tried first, and nothing
    // is read back - the call only enqueues (no host synchronisation), so consecutive steps run back to back on the GPU.
    int solve_enqueue(const SolveRequest& r, cudaStream_t st);
    // anchors (seed[i] == i or out of range) cold, then every other sample from its anchor's certified active set
    int solve_seeded(const SolveRequest& r, cudaStream_t st, SolveCounts* counts = nullptr);
};

}  // namespace carmpc
