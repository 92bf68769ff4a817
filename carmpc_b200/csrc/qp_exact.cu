// Float64 fallback of the batched QP solver: the last resort for the few samples (none on most grids, a few hundred per
// 10^6 for RoadMultipleCarsEnv, whose x-y coupled rows make degenerate vertices common) that leave the second float32
// ADMM pass + polish without a decision the library can PROVE:
//   - "solved" by the float32 ADMM but the float64 polish found no KKT certificate (a barely infeasible state looks
//     converged at float32 tolerances: residual 3e-5 against an infeasibility of 1e-4), or
//   - out of iterations.
// Nothing leaves the library as CARMPC_QP_SOLVED without a float64 KKT certificate, and nothing as
// CARMPC_QP_INFEASIBLE without a float64 Farkas certificate; what even this kernel cannot settle is CARMPC_QP_MAX_ITER.
//
// One warp per sample runs the same ADMM (single-vector form  v = 2 clip(w) - w ; x~ = x~0 + rho K^-1 A' v ; z = A x~ ;
// w += alpha (z - clip(w)),  A = [Gs; diag(lam)] equilibrated as in qp_setup.cu) in float64 to a 1e-9 residual, starting
// from the sample's float32 ADMM state; at every check the dual iterate y = E (w - clip(w)), completed with box
// multipliers y_b = -G'y so that A'y = 0 holds exactly, is evaluated as a Farkas certificate (the test of
// farkas_kernel, qp_polish.cu).  A converged sample hands its active set (the signs of w against its bounds) to one
// more float64 polish, which certifies it or leaves it undecided.
#include <math.h>
#include <string.h>

#include <algorithm>

#include "qp_internal.cuh"

namespace carmpc {

namespace {

constexpr int kExactThreads = 128;
constexpr int kExactCheck = 25;
constexpr double kExactEps = 1e-9;

__device__ __forceinline__ double wsum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ double wmax(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
__device__ __forceinline__ double clampd(double w, double lo, double hi) { return fmin(fmax(w, lo), hi); }

// samples of `list` that are still unproven after the second pass: out of iterations, "infeasible" without a float64
// certificate, or "solved" without a KKT certificate
__global__ void collect_unproven_kernel(const int* __restrict__ list, int count, const int* __restrict__ count_dev,
                                        const int* __restrict__ status, const int8_t* __restrict__ polished,
                                        int* __restrict__ out, int* __restrict__ n_out) {
    if (count_dev != nullptr) count = min(count, *count_dev);
    for (int q = blockIdx.x * blockDim.x + threadIdx.x; q < count; q += gridDim.x * blockDim.x) {
        const int s = list[q];
        const int st = status[s];
        if (st == CARMPC_QP_MAX_ITER || st == kStatusNeedsMoreAdmm || (st == CARMPC_QP_SOLVED && polished[s] == 0))
            out[atomicAdd(n_out, 1)] = s;
    }
}

// sum_k M[k * ld + col] * x[k], four independent chains (the tables come from L1 / L2: latency, not throughput)
__device__ __forceinline__ double col_dot(const double* __restrict__ M, int ld, int col, const double* x, int len) {
    double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
    const double* p = M + col;
    int k = 0;
    for (; k + 4 <= len; k += 4) {
        const double a0 = p[(size_t)k * ld], a1 = p[(size_t)(k + 1) * ld], a2 = p[(size_t)(k + 2) * ld], a3 = p[(size_t)(k + 3) * ld];
        s0 += a0 * x[k]; s1 += a1 * x[k + 1]; s2 += a2 * x[k + 2]; s3 += a3 * x[k + 3];
    }
    for (; k < len; ++k) s0 += p[(size_t)k * ld] * x[k];
    return (s0 + s1) + (s2 + s3);
}

// per-warp workspace in shared memory
struct ExactWs {
    double *w, *v, *h, *l, *yp, *r, *xt, *xt0;
    __device__ static size_t doubles(int n, int mt) { return 5 * (size_t)mt + 3 * (size_t)n; }
    __device__ ExactWs(double* base, int n, int mt) {
        w = base; v = w + mt; h = v + mt; l = h + mt; yp = l + mt; r = yp + mt; xt = r + n; xt0 = xt + n;
    }
};

// bounds of this sample in equilibrated units, the float32 ADMM state as the start point, x~0 = -K^-1 q_s
__device__ __forceinline__ void exact_setup(const PolishTables& T, const ExactTables& E, const ExactWs& S, const double (&x0)[4],
                                            const double (&dx)[4], double cd, const float* warm, int lane) {
    const int n = T.n, m = T.m, mt = T.mt;
    for (int i = lane; i < mt; i += 32) {
        double hi = T.hi[i], lo = T.lo[i], e;
        if (i < m) {
            const double* gx = T.Gx + (size_t)i * 4;
            const double shift = gx[0] * x0[0] + gx[1] * x0[1] + gx[2] * x0[2] + gx[3] * x0[3] + T.Gc[i] * cd;
            e = T.Eg[i];
            hi -= shift; lo -= shift;
        } else {
            e = E.Eb[i - m];
        }
        S.h[i] = isinf(hi) ? INFINITY : e * hi;
        S.l[i] = isinf(lo) ? -INFINITY : e * lo;
        const double w0 = (double)warm[i];
        S.w[i] = isfinite(w0) ? w0 : 0.0;
    }
    for (int k = lane; k < n; k += 32) {               // r <- scaled linear term  c D F dx
        const double* f = T.F + (size_t)k * 4;
        S.r[k] = E.cs * E.D[k] * (f[0] * dx[0] + f[1] * dx[1] + f[2] * dx[2] + f[3] * dx[3]);
    }
    __syncwarp();
    for (int j = lane; j < n; j += 32) S.xt0[j] = -col_dot(E.Kinv, n, j, S.r, n);      // K^-1 symmetric: column walk is coalesced
    __syncwarp();
}

// one ADMM iteration in float64; with `measure` also the residual norms of the f32 kernel's stopping test
__device__ __forceinline__ void exact_step(const PolishTables& T, const ExactTables& E, const ExactWs& S, int lane, bool measure,
                                           double& res, double& nrm) {
    const int n = T.n, m = T.m, mt = T.mt;
    for (int i = lane; i < mt; i += 32) { const double wi = S.w[i]; S.v[i] = 2.0 * clampd(wi, S.l[i], S.h[i]) - wi; }
    __syncwarp();
    for (int j = lane; j < n; j += 32) S.r[j] = E.lam[j] * S.v[m + j] + col_dot(E.Gs, n, j, S.v, m);
    __syncwarp();
    for (int j = lane; j < n; j += 32) S.xt[j] = S.xt0[j] + E.rho * col_dot(E.Kinv, n, j, S.r, n);
    __syncwarp();
    for (int i = lane; i < mt; i += 32) {
        const double z = i < m ? col_dot(E.GsT, m, i, S.xt, n) : E.lam[i - m] * S.xt[i - m];
        const double w0 = S.w[i], c0 = clampd(w0, S.l[i], S.h[i]);
        const double w1 = w0 + E.alpha * (z - c0), c1 = clampd(w1, S.l[i], S.h[i]);
        S.w[i] = w1;
        if (measure) {
            const double einv = 1.0 / (i < m ? T.Eg[i] : E.Eb[i - m]);
            res = fmax(res, fmax(fabs(z - c1), fabs(c1 - c0)) * einv);
            nrm = fmax(nrm, fmax(fabs(z), fabs(c1)) * einv);
        }
    }
    __syncwarp();
}

// scaled dual of the general rows: y = w - clip(w)
__device__ __forceinline__ void exact_dual(const ExactWs& S, double* y, int m, int lane) {
    for (int i = lane; i < m; i += 32) { const double wi = S.w[i]; y[i] = wi - clampd(wi, S.l[i], S.h[i]); }
    __syncwarp();
}

// Farkas test of the direction d (scaled units, general rows; in S.v): multipliers of the unscaled rows y = Eg d (entries
// that would need an infinite bound are dropped), box multipliers y_b = -G'y, so that A'y = 0 holds exactly; infeasible
// iff the support value  b'y + box support  is negative.  Overwrites S.v with y.
__device__ __forceinline__ bool exact_farkas(const PolishTables& T, const ExactWs& S, int lane) {
    const int n = T.n, m = T.m;
    double c0 = 0.0, a0 = 0.0;
    for (int i = lane; i < m; i += 32) {
        double d = S.v[i];
        if ((d > 0.0 && isinf(S.h[i])) || (d < 0.0 && isinf(S.l[i]))) d = 0.0;
        const double yu = T.Eg[i] * d;
        S.v[i] = yu;
        if (yu != 0.0) {
            const double bound = (yu > 0.0 ? S.h[i] : S.l[i]) / T.Eg[i];      // unscaled bound of this sample (shifts included)
            c0 += bound * yu; a0 += fabs(bound * yu);
        }
    }
    __syncwarp();
    for (int j = lane; j < n; j += 32) {
        const double yb = -col_dot(T.G, n, j, S.v, m);
        if (yb != 0.0) {
            const double t = (yb > 0.0 ? T.hi[m + j] : T.lo[m + j]) * yb;
            c0 += t; a0 += fabs(t);
        }
    }
    c0 = wsum(c0); a0 = wsum(a0);
    __syncwarp();
    return isfinite(c0) && isfinite(a0) && a0 > 0.0 && c0 < -1e-9 * a0;
}

// Certificate row of a ray exact_farkas accepted (y in S.v): the general part in the caller's orientation, the box part by
// the same expression the test used, zeros on the u-independent rows.
__device__ __forceinline__ void store_ray(const PolishTables& T, const ExactWs& S, double* row, int lane) {
    const int n = T.n, m = T.m, mt = T.mt;
    for (int i = lane; i < m; i += 32) row[i] = T.rsign[i] * S.v[i];
    for (int j = lane; j < n; j += 32) row[m + j] = -col_dot(T.G, n, j, S.v, m);
    for (int k = lane; k < T.kpre; k += 32) row[mt + k] = 0.0;
}

// ---- verification of the float32 "infeasible" verdicts -----------------------------------------------------------------------
// The float32 ADMM certifies infeasibility with the dual INCREMENT of one iteration (qp_admm.cu) under a 1e-4 relative
// margin.  Here the same increment is recomputed in float64 - one ADMM iteration from the sample's stored state - and
// must pass the exact test; a violated u-independent row is a proof by itself.  Unverified samples re-enter the second
// pass (status kStatusNeedsMoreAdmm, appended to `failed`).
struct VerifyArgs {
    const int* list; int count; const int* count_dev;
    const double* x0; int64_t stride; const double* cdist; double xref[4];
    const float* warm; int* status;
    const double* Px; const double* Pc; const double* pre_lo; const double* pre_hi; int kpre;
    int* failed; int* n_failed;
    unsigned long long* row_proofs;     // nullable counter: verdicts proven by a single row
    double* cert;                       // nullable [batch][mt + kpre]: the proof of every verified sample
};

// CERT: the certificate stores are a separate instantiation, so that a solve without certificates runs the same code as before
template <bool CERT>
__global__ void __launch_bounds__(kExactThreads) verify_kernel(const PolishTables T, const ExactTables E, const VerifyArgs A) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int n = T.n, m = T.m, mt = T.mt;
    const ExactWs S(reinterpret_cast<double*>(smem_raw) + (size_t)warp * ExactWs::doubles(n, mt), n, mt);
    const int gw = blockIdx.x * (kExactThreads / 32) + warp, nw = gridDim.x * (kExactThreads / 32);
    const int v_count = A.count_dev != nullptr ? min(*A.count_dev, A.count) : A.count;
    for (int q = gw; q < v_count; q += nw) {
        const int sample = A.list ? A.list[q] : q;
        if (A.status[sample] != CARMPC_QP_INFEASIBLE) continue;
        double x0[4], dx[4];
#pragma unroll
        for (int c = 0; c < 4; ++c) { x0[c] = A.x0[(size_t)c * A.stride + sample]; dx[c] = x0[c] - A.xref[c]; }
        const double cd = A.cdist ? A.cdist[sample] : 0.0;
        bool pre_ok = isfinite(x0[0]) && isfinite(x0[1]) && isfinite(x0[2]) && isfinite(x0[3]) && isfinite(cd);
        for (int k = 0; k < A.kpre && pre_ok; ++k) {
            const double v = A.Px[k * 4 + 0] * x0[0] + A.Px[k * 4 + 1] * x0[1] + A.Px[k * 4 + 2] * x0[2] + A.Px[k * 4 + 3] * x0[3] +
                             A.Pc[k] * cd;
            pre_ok = v <= A.pre_hi[k] && v >= A.pre_lo[k];
        }
        if (!pre_ok) {                                                 // infeasible whatever u is: nothing to verify
            if (CERT) store_pre_certificate(A.cert + (size_t)sample * (mt + T.kpre), mt, T.kpre, A.Px, A.Pc, A.pre_lo, A.pre_hi, x0, cd, lane);
            continue;
        }
        __syncwarp();
        // single-row certificates: the bound of a row lies outside what G_i u can reach over the input box
        bool row_proof = false;
        int proof_row = -1;                                            // the first such row of this lane, +-(i + 1)
        for (int i = lane; i < m; i += 32) {
            const double* gx = T.Gx + (size_t)i * 4;
            const double t0 = gx[0] * x0[0], t1 = gx[1] * x0[1], t2 = gx[2] * x0[2], t3 = gx[3] * x0[3], t4 = T.Gc[i] * cd;
            const double shift = t0 + t1 + t2 + t3 + t4;
            const double hi = T.hi[i], lo = T.lo[i];
            const double slop = 1e-12 * (fabs(t0) + fabs(t1) + fabs(t2) + fabs(t3) + fabs(t4) + E.rowabs[i] + (isinf(hi) ? 0.0 : fabs(hi)) +
                                         (isinf(lo) ? 0.0 : fabs(lo)));
            row_proof = row_proof || (hi - shift < E.rowmin[i] - slop) || (lo - shift > E.rowmax[i] + slop);
            if (CERT && row_proof && proof_row == -1) proof_row = hi - shift < E.rowmin[i] - slop ? i + 1 : -(i + 1);
        }
        if (__any_sync(0xffffffffu, row_proof)) {
            if (lane == 0 && A.row_proofs) atomicAdd(A.row_proofs, 1ull);
            if (CERT) {
                // y = +-1 on that row, box part -G_i' y: the support value is (hi - shift) - rowmin (or rowmax - (lo - shift))
                const unsigned proof_lanes = __ballot_sync(0xffffffffu, row_proof);
                const int pr = __shfl_sync(0xffffffffu, proof_row, __ffs(proof_lanes) - 1);
                const int i = abs(pr) - 1;
                const double yi = pr > 0 ? 1.0 : -1.0;
                double* row = A.cert + (size_t)sample * (mt + T.kpre);
                for (int e = lane; e < m; e += 32) row[e] = e == i ? T.rsign[i] * yi : 0.0;
                for (int j = lane; j < n; j += 32) row[m + j] = -T.G[(size_t)i * n + j] * yi;
                for (int k = lane; k < T.kpre; k += 32) row[mt + k] = 0.0;
            }
            continue;
        }
        exact_setup(T, E, S, x0, dx, cd, A.warm + (size_t)sample * mt, lane);
        bool proven = false;
        for (int round = 0; round < 3 && !proven; ++round) {           // the increment of the 1st, 2nd, 4th iteration from the state
            exact_dual(S, S.yp, m, lane);
            double res = 0.0, nrm = 0.0;
            for (int k = 0; k < (round < 2 ? 1 : 2); ++k) exact_step(T, E, S, lane, false, res, nrm);
            for (int i = lane; i < m; i += 32) { const double wi = S.w[i]; S.v[i] = (wi - clampd(wi, S.l[i], S.h[i])) - S.yp[i]; }
            __syncwarp();
            proven = exact_farkas(T, S, lane);
        }
        if (CERT) {
            double* row = A.cert + (size_t)sample * (mt + T.kpre);
            if (proven) store_ray(T, S, row, lane);
            else for (int e = lane; e < mt + T.kpre; e += 32) row[e] = 0.0;      // a proof stored earlier did not hold up
        }
        if (!proven && lane == 0) {
            A.status[sample] = kStatusNeedsMoreAdmm;
            A.failed[atomicAdd(A.n_failed, 1)] = sample;
        }
    }
}

struct ExactArgs {
    const int* list;
    const int* count_dev;
    int count_max;
    int max_iter;
    const double* x0; int64_t stride; const double* cdist; double xref[4];
    const float* warm;            // [batch][mt] float32 ADMM state (start point), logical row order
    int8_t* sign;                 // [batch][mt] out: active-set guess for the polish
    int* status;                  // out: SOLVED (to be certified by the polish), INFEASIBLE, MAX_ITER
    int* iters;                   // += float64 iterations
    double* u0; double* objective; double* u_full; int8_t* polished;
    unsigned long long* stats;
    unsigned long long* total_iters;
    double* cert;                 // nullable [batch][mt + kpre]: the ray of every sample proven infeasible here
};

template <bool CERT>
__global__ void __launch_bounds__(kExactThreads) exact_kernel(const PolishTables T, const ExactTables E, const ExactArgs A) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int n = T.n, m = T.m, mt = T.mt;
    const ExactWs S(reinterpret_cast<double*>(smem_raw) + (size_t)warp * ExactWs::doubles(n, mt), n, mt);
    const int count = min(*A.count_dev, A.count_max);
    const int gw = blockIdx.x * (kExactThreads / 32) + warp, nw = gridDim.x * (kExactThreads / 32);
    const double NaN = __longlong_as_double(0x7ff8000000000000ll);
    for (int q = gw; q < count; q += nw) {
        const int sample = A.list[q];
        double x0[4], dx[4];
#pragma unroll
        for (int c = 0; c < 4; ++c) { x0[c] = A.x0[(size_t)c * A.stride + sample]; dx[c] = x0[c] - A.xref[c]; }
        const double cd = A.cdist ? A.cdist[sample] : 0.0;
        __syncwarp();
        exact_setup(T, E, S, x0, dx, cd, A.warm + (size_t)sample * mt, lane);
        exact_dual(S, S.yp, m, lane);
        int verdict = CARMPC_QP_MAX_ITER, it = 0;
        double res = 0.0, nrm = 0.0;
        while (it < A.max_iter) {
            res = 0.0; nrm = 0.0;
            for (int sub = 0; sub < kExactCheck; ++sub, ++it) exact_step(T, E, S, lane, sub == kExactCheck - 1, res, nrm);
            res = wmax(res); nrm = wmax(nrm);
            if (!(res == res)) break;                               // NaN state: undecided
            if (res <= kExactEps * (1.0 + nrm)) { verdict = CARMPC_QP_SOLVED; break; }
            // certificate from the dual increment over the last kExactCheck iterations, then from the dual itself (which a
            // long run of an infeasible problem ends up dominated by)
            for (int i = lane; i < m; i += 32) {
                const double wi = S.w[i], y = wi - clampd(wi, S.l[i], S.h[i]);
                S.v[i] = y - S.yp[i];
                S.yp[i] = y;
            }
            __syncwarp();
            if (exact_farkas(T, S, lane)) { verdict = CARMPC_QP_INFEASIBLE; break; }
            for (int i = lane; i < m; i += 32) S.v[i] = S.yp[i];
            __syncwarp();
            if (exact_farkas(T, S, lane)) { verdict = CARMPC_QP_INFEASIBLE; break; }
        }
        // ---- hand over ----
        // Out of iterations but close (a degenerate vertex: linearly dependent active rows make the dual drift for ever while
        // the primal iterate is already within 1e-6 of the optimum): the active set still goes to the polish, which
        // either certifies an exact KKT point or leaves the sample undecided.
        if (verdict == CARMPC_QP_MAX_ITER && res == res && res <= 1e-5 * (1.0 + nrm)) verdict = CARMPC_QP_SOLVED;
        if (verdict == CARMPC_QP_SOLVED) {
            for (int i = lane; i < mt; i += 32) {
                const double wi = S.w[i];
                A.sign[(size_t)sample * mt + i] = (int8_t)((wi > S.h[i]) - (wi < S.l[i]));
            }
        }
        if (CERT && verdict == CARMPC_QP_INFEASIBLE) store_ray(T, S, A.cert + (size_t)sample * (mt + T.kpre), lane);
        if (verdict != CARMPC_QP_SOLVED && A.u_full) for (int j = lane; j < n; j += 32) A.u_full[(size_t)sample * n + j] = NaN;
        if (lane == 0) {
            A.status[sample] = verdict;
            if (A.iters) A.iters[sample] += it;
            if (A.total_iters) atomicAdd(A.total_iters, (unsigned long long)it);
            if (verdict != CARMPC_QP_SOLVED) {
                if (A.u0) { A.u0[sample] = NaN; A.u0[A.stride + sample] = NaN; }
                if (A.objective) A.objective[sample] = verdict == CARMPC_QP_INFEASIBLE ? INFINITY : NaN;
                if (A.polished) A.polished[sample] = 0;
                if (A.stats) atomicAdd(A.stats + (verdict == CARMPC_QP_INFEASIBLE ? 18 : 19), 1ull);
            }
        }
    }
}

static size_t exact_smem(int n, int mt) { return sizeof(double) * (kExactThreads / 32) * (5 * (size_t)mt + 3 * (size_t)n); }

}  // namespace

// After the second pass: everything in `d_list` that is still unproven goes through the float64 ADMM; converged samples
// get one more polish (strict: no certificate -> CARMPC_QP_MAX_ITER).  Returns the number of samples handled.
int exact_fallback(QPHandle* q, const PolishBatch& b, const int* d_list, int count, const int* d_count, float* d_warm,
                   int* d_iters, cudaStream_t st, int* h_handled) {
    *h_handled = 0;
    if (count <= 0) return CARMPC_OK;
    int* n_unproven = q->ws_counters + kCntUnproven;
    CARMPC_CUDA(cudaMemsetAsync(n_unproven, 0, sizeof(int), st));
    collect_unproven_kernel<<<std::min((count + 255) / 256, 64), 256, 0, st>>>(d_list, count, d_count, b.status, b.polished,
                                                                          q->ws_unproven, n_unproven);
    int n = 0;
    if (d_count == nullptr) {
        CARMPC_CUDA(cudaMemcpyAsync(&n, n_unproven, sizeof(int), cudaMemcpyDeviceToHost, st));
        CARMPC_CUDA(cudaStreamSynchronize(st));
        if (n == 0) return CARMPC_OK;
    } else {
        n = std::min(count, 4 * q->sm * 2);        // device-sized: a fixed small grid, the kernels read the count themselves
    }
    *h_handled = n;
    ExactArgs a;
    memset(&a, 0, sizeof(a));
    a.list = q->ws_unproven; a.count_dev = n_unproven; a.count_max = d_count == nullptr ? n : count;
    a.x0 = b.x0; a.stride = b.stride; a.cdist = b.cdist;
    for (int c = 0; c < 4; ++c) a.xref[c] = b.xref[c];
    a.warm = d_warm; a.sign = q->ws_sign; a.status = b.status; a.iters = d_iters;
    a.u0 = b.u0; a.objective = b.objective; a.u_full = b.u_full; a.polished = b.polished;
    a.stats = b.stats; a.total_iters = q->ws_total_iters; a.cert = b.cert;
    const int mt = q->polish.mt, nn = q->polish.n;
    // iteration budget: ~4e8 multiply-adds per sample (5000 iterations at N = 20, ~2600 at N = 80)
    const double macs = 2.0 * q->polish.m * nn + (double)nn * nn;
    a.max_iter = (int)std::max(1000.0, std::min(5000.0, 4.0e8 / std::max(1.0, macs)));
    const size_t smem = exact_smem(nn, mt);
    void (*kernel)(const PolishTables, const ExactTables, const ExactArgs) = a.cert ? exact_kernel<true> : exact_kernel<false>;
    { const int rc = kernel_config(reinterpret_cast<const void*>(kernel), kExactThreads, smem, nullptr); if (rc != CARMPC_OK) return rc; }
    const int blocks = std::max(1, std::min((n + 3) / 4, q->sm * 2));
    kernel<<<blocks, kExactThreads, smem, st>>>(q->polish, q->exact, a);
    CARMPC_CUDA(cudaGetLastError());
    // one more float64 polish from the float64 active sets; strict: an uncertified sample becomes "undecided"
    PolishBatch pb = b;
    pb.idx_list = q->ws_unproven; pb.count = d_count == nullptr ? n : count; pb.count_dev = d_count == nullptr ? nullptr : n_unproven;
    pb.n_failed = q->ws_counters + kCntExactFinal; pb.final_pass = 2; pb.rounds = 40;
    return polish_launch(q, pb, st);
}

int farkas_verify_launch(QPHandle* q, const PolishBatch& b, const int* d_list, int count, const int* d_count,
                         const float* d_warm, int* d_failed, int* d_n_failed, cudaStream_t st) {
    if (count <= 0) return CARMPC_OK;
    VerifyArgs a;
    memset(&a, 0, sizeof(a));
    a.list = d_list; a.count = count; a.count_dev = d_count; a.x0 = b.x0; a.stride = b.stride; a.cdist = b.cdist;
    for (int c = 0; c < 4; ++c) a.xref[c] = b.xref[c];
    a.warm = d_warm; a.status = b.status;
    a.Px = q->admm.Px; a.Pc = q->admm.Pc; a.pre_lo = q->admm.pre_lo; a.pre_hi = q->admm.pre_hi; a.kpre = q->admm.kpre;
    a.failed = d_failed; a.n_failed = d_n_failed; a.cert = b.cert;
    const size_t smem = exact_smem(q->polish.n, q->polish.mt);
    int per_sm = 0;
    void (*kernel)(const PolishTables, const ExactTables, const VerifyArgs) = a.cert ? verify_kernel<true> : verify_kernel<false>;
    { const int rc = kernel_config(reinterpret_cast<const void*>(kernel), kExactThreads, smem, &per_sm); if (rc != CARMPC_OK) return rc; }
    const int blocks = (int)std::max<int64_t>(1, std::min<int64_t>((count + 3) / 4, (int64_t)q->sm * std::max(per_sm, 1)));
    kernel<<<blocks, kExactThreads, smem, st>>>(q->polish, q->exact, a);
    CARMPC_CUDA(cudaGetLastError());
    return CARMPC_OK;
}

}  // namespace carmpc
