// Independent float64 check of QP certificates (carmpc_qp_checker_create / carmpc_qp_check).
//
// The checker takes a QP in the general two-sided form
//       min 1/2 u'Hu + (F (x0 - xref))'u     lo - Gx x0 - Gc c <= G u <= hi - Gx x0 - Gc c ,   lb <= u <= ub
// with R general rows, as the caller states it (a one-sided reference stack is lo = -inf).  It shares nothing with the
// solver's setup: no equilibration, no row merging, no chain analysis, no padding, no solver handle.  One warp per
// sample; G' (n x R) sits in shared memory when it fits and is read through L2 otherwise.
//
// A certificate row has R + n entries (general rows, then box rows); positive means "against the upper bound", negative
// "against the lower bound".  Per sample, 4 doubles:
//   status 0 (multipliers lam):  [0] primal violation, per row relative to max(1, sum_j |G_ij u_j|) (box: max(1, |u_j|))
//                                [1] stationarity |H u + q + G' lam_g + lam_b|_inf relative to max(1, |H u|_inf, |q|_inf),
//                                    the size of the gradient's two terms (an unconstrained optimum cancels them)
//                                [2] largest |lam_i| against an infinite bound, relative to max(1, |lam|_inf)
//                                [3] complementarity max |lam_i| |slack_i| on the side lam_i pushes against, relative to
//                                    max(1, |lam|_inf) max(1, sum_j |G_ij u_j|)
//   status 1 (Farkas ray y):     the box part is completed here, y_b = -G' y_g, so that it does not depend on the caller's
//                                [0] support value  sum_i (y_i+ (hi_i - s_i) - y_i- (lo_i - s_i)) + box support of y_b
//                                [1] its rounding scale (see kSupportMargin)
//                                [2] |G' y_g + y_b|_inf of the caller's box part, relative to max_j sum_i |G_ij y_i|
//                                [3] wrong-sign mass: sum of |y_i| (completed box part included) against an infinite bound
//                                The ray proves infeasibility iff [3] == 0 and [0] < -kSupportMargin [1].
//   status 2 (undecided):        NaN.
#include <float.h>
#include <math.h>
#include <string.h>

#include <algorithm>
#include <vector>

#include "common.cuh"

namespace carmpc {

namespace {

constexpr int kCheckThreads = 256;
constexpr int kCheckMaxN = 160;
constexpr int kCheckMaxR = 16000;
constexpr size_t kCheckSmemGT = 150 * 1024;     // G' stays in shared memory up to this size (N = 20: 56 KB; N = 80: 763 KB)

// Rounding margin of the support value.  Every sum below is a float64 dot product; a dot product of K terms has an error
// of at most gamma_K sum |terms|, gamma_K = K u / (1 - K u), u = 2^-53, whatever the order and FMA contraction.  The
// support is a sum of R + n terms y_i (bound_i - s_i) and y_b,j bound_j, with s_i a 5-term sum and y_b,j = -sum_i G_ij y_i an
// R-term sum.  The computed y_b leaves G'y_g + y_b = e with |e_j| <= gamma_R sum_i |G_ij y_i|, which a feasible u turns
// into e'u <= sum_j |e_j| max(|lb_j|, |ub_j|).  So the exact support of the ray (y_g, computed y_b) plus that slack
// differs from the computed value by at most gamma_K * scale, K = 2R + n + 8, with
//     scale = sum_i |y_i| (|bound_i| + sum_c |Gx_ic x0_c| + |Gc_i c|) + sum_j (sum_i |G_ij y_i|) max(|lb_j|, |ub_j|)
// (an infinite box side under a non-zero column makes it infinite: no proof).  R <= 16000 and n <= 160 give K <= 32168 and
// gamma_K < 3.58e-12: a computed support below -4e-12 scale is negative in exact arithmetic, and the ray is a proof.
constexpr double kSupportMargin = 4e-12;

struct CheckTables {
    const double* H;     // [n][n]
    const double* F;     // [n][4]
    const double* G;     // [R][n]
    const double* GT;    // [n][R]
    const double* Gx;    // [R][4]
    const double* Gc;    // [R]
    const double* lo;    // [R]
    const double* hi;
    const double* lb;    // [n]
    const double* ub;
    int n, R;
    int gt_smem;
};

struct CheckArgs {
    const double* x0; int64_t batch; const double* c; double xref[4];
    const int32_t* status; const double* u_full; const double* cert; double* resid;
};

__device__ __forceinline__ double cwmax(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
__device__ __forceinline__ double cwsum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

__global__ void __launch_bounds__(kCheckThreads) qp_check_kernel(const CheckTables T, const CheckArgs A) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    constexpr int kCols = kCheckMaxN / 32;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int n = T.n, R = T.R;
    double* gts = reinterpret_cast<double*>(smem_raw);
    const size_t gt_doubles = T.gt_smem ? (size_t)n * R : 0;
    if (T.gt_smem)
        for (size_t e = threadIdx.x; e < gt_doubles; e += blockDim.x) gts[e] = T.GT[e];
    __syncthreads();
    const double* GT = T.gt_smem ? gts : T.GT;
    double* us = gts + gt_doubles + (size_t)warp * n;
    const double NaN = __longlong_as_double(0x7ff8000000000000ll);
    const int64_t gw = (int64_t)blockIdx.x * (kCheckThreads / 32) + warp, nw = (int64_t)gridDim.x * (kCheckThreads / 32);
    for (int64_t s = gw; s < A.batch; s += nw) {
        const int st = A.status[s];
        double* out = A.resid + s * 4;
        if (st != CARMPC_QP_SOLVED && st != CARMPC_QP_INFEASIBLE) {
            if (lane < 4) out[lane] = NaN;
            continue;
        }
        double x0[4], dx[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) { x0[k] = A.x0[(size_t)k * A.batch + s]; dx[k] = x0[k] - A.xref[k]; }
        const double cd = A.c ? A.c[s] : 0.0;
        const double* crow = A.cert + (size_t)s * (R + n);
        // G' y_g per column (this lane's columns j = lane + 32 t), in row order; only rows with a non-zero entry contribute
        double acc[kCols], aacc[kCols];
#pragma unroll
        for (int t = 0; t < kCols; ++t) { acc[t] = 0.0; aacc[t] = 0.0; }
        double ymax = 0.0;
        for (int i0 = 0; i0 < R; i0 += 32) {
            const double yi = i0 + lane < R ? crow[i0 + lane] : 0.0;
            ymax = fmax(ymax, fabs(yi));
            unsigned mask = __ballot_sync(0xffffffffu, yi != 0.0);
            while (mask) {
                const int src = __ffs(mask) - 1;
                mask &= mask - 1;
                const double y = __shfl_sync(0xffffffffu, yi, src);
                const double* row = T.G + (size_t)(i0 + src) * n;
#pragma unroll
                for (int t = 0; t < kCols; ++t) {
                    const int j = lane + 32 * t;
                    if (j < n) { const double p = row[j] * y; acc[t] += p; aacc[t] += fabs(p); }
                }
            }
        }
        if (st == CARMPC_QP_SOLVED) {
            for (int j = lane; j < n; j += 32) us[j] = A.u_full[(size_t)s * n + j];
            __syncwarp();
            double lmax = ymax;
            for (int j = lane; j < n; j += 32) lmax = fmax(lmax, fabs(crow[R + j]));
            lmax = fmax(1.0, cwmax(lmax));
            double primal = 0.0, stat_r = 0.0, stat_s = 1.0, wrong = 0.0, compl_ = 0.0;
#pragma unroll
            for (int t = 0; t < kCols; ++t) {
                const int j = lane + 32 * t;
                if (j >= n) continue;
                double hu = 0.0;
                for (int k = 0; k < n; ++k) hu += T.H[(size_t)j * n + k] * us[k];
                const double* f = T.F + (size_t)j * 4;
                const double q = f[0] * dx[0] + f[1] * dx[1] + f[2] * dx[2] + f[3] * dx[3];
                const double lamb = crow[R + j], uj = us[j];
                stat_r = fmax(stat_r, fabs(hu + q + acc[t] + lamb));
                stat_s = fmax(stat_s, fmax(fabs(hu), fabs(q)));
                const double sc = fmax(1.0, fabs(uj));
                primal = fmax(primal, fmax(0.0, fmax(uj - T.ub[j], T.lb[j] - uj)) / sc);
                if (lamb > 0.0) {
                    if (isinf(T.ub[j])) wrong = fmax(wrong, lamb); else compl_ = fmax(compl_, lamb * fabs(T.ub[j] - uj) / sc);
                } else if (lamb < 0.0) {
                    if (isinf(T.lb[j])) wrong = fmax(wrong, -lamb); else compl_ = fmax(compl_, -lamb * fabs(uj - T.lb[j]) / sc);
                } else if (lamb != lamb) {
                    wrong = NaN;
                }
            }
            for (int i = lane; i < R; i += 32) {
                double gu = 0.0, ga = 0.0;
                for (int k = 0; k < n; ++k) { const double p = GT[(size_t)k * R + i] * us[k]; gu += p; ga += fabs(p); }
                const double* gx = T.Gx + (size_t)i * 4;
                const double sh = gx[0] * x0[0] + gx[1] * x0[1] + gx[2] * x0[2] + gx[3] * x0[3] + (T.Gc ? T.Gc[i] * cd : 0.0);
                const double his = T.hi[i] - sh, los = T.lo[i] - sh, sc = fmax(1.0, ga);
                primal = fmax(primal, fmax(0.0, fmax(gu - his, los - gu)) / sc);
                const double l = crow[i];
                if (l > 0.0) {
                    if (isinf(T.hi[i])) wrong = fmax(wrong, l); else compl_ = fmax(compl_, l * fabs(his - gu) / sc);
                } else if (l < 0.0) {
                    if (isinf(T.lo[i])) wrong = fmax(wrong, -l); else compl_ = fmax(compl_, -l * fabs(gu - los) / sc);
                } else if (l != l) {
                    wrong = NaN;
                }
            }
            primal = cwmax(primal); stat_r = cwmax(stat_r); stat_s = cwmax(stat_s); wrong = cwmax(wrong); compl_ = cwmax(compl_);
            // fmax drops NaN: a non-finite u or multiplier must not pass
            bool finite = true;
            for (int j = lane; j < n; j += 32) finite = finite && isfinite(us[j]) && isfinite(crow[R + j]);
            for (int i = lane; i < R; i += 32) finite = finite && isfinite(crow[i]);
            finite = __all_sync(0xffffffffu, finite);
            if (lane == 0) {
                out[0] = finite ? primal : NaN;
                out[1] = finite ? stat_r / stat_s : NaN;
                out[2] = finite ? wrong / lmax : NaN;
                out[3] = finite ? compl_ / lmax : NaN;
            }
            __syncwarp();
        } else {
            double sup = 0.0, scale = 0.0, res = 0.0, amax = 0.0, wrong = 0.0;
#pragma unroll
            for (int t = 0; t < kCols; ++t) {
                const int j = lane + 32 * t;
                if (j >= n) continue;
                const double yb = -acc[t];
                res = fmax(res, fabs(acc[t] + crow[R + j]));
                amax = fmax(amax, aacc[t]);
                if (aacc[t] != 0.0) {
                    const double ub = T.ub[j], lb = T.lb[j];
                    scale += aacc[t] * fmax(fabs(ub), fabs(lb));
                }
                if (yb > 0.0) { if (isinf(T.ub[j])) wrong += yb; else sup += yb * T.ub[j]; }
                else if (yb < 0.0) { if (isinf(T.lb[j])) wrong -= yb; else sup += yb * T.lb[j]; }
            }
            for (int i = lane; i < R; i += 32) {
                const double y = crow[i];
                if (y == 0.0) continue;
                const double* gx = T.Gx + (size_t)i * 4;
                const double t0 = gx[0] * x0[0], t1 = gx[1] * x0[1], t2 = gx[2] * x0[2], t3 = gx[3] * x0[3];
                const double t4 = T.Gc ? T.Gc[i] * cd : 0.0;
                const double bound = y > 0.0 ? T.hi[i] : T.lo[i];
                if (isinf(bound) || y != y) { wrong += fabs(y); continue; }
                sup += y * (bound - (t0 + t1 + t2 + t3 + t4));
                scale += fabs(y) * (fabs(bound) + fabs(t0) + fabs(t1) + fabs(t2) + fabs(t3) + fabs(t4));
            }
            sup = cwsum(sup); scale = cwsum(scale); wrong = cwsum(wrong);
            res = cwmax(res); amax = cwmax(amax);
            if (lane == 0) {
                out[0] = sup;
                out[1] = scale;
                out[2] = res / fmax(amax, DBL_MIN);
                out[3] = wrong;
            }
            __syncwarp();
        }
    }
}

struct QPCheckHandle : HandleBase {
    CheckTables t{};
    std::vector<void*> allocations;
    bool host_only = false;
    ~QPCheckHandle() override { for (void* p : allocations) cudaFree(p); }
};

int upload_doubles(QPCheckHandle* q, const std::vector<double>& v, const double** dst) {
    void* d = nullptr;
    CARMPC_CUDA(cudaMalloc(&d, sizeof(double) * std::max<size_t>(v.size(), 1)));
    q->allocations.push_back(d);
    if (!v.empty()) CARMPC_CUDA(cudaMemcpy(d, v.data(), sizeof(double) * v.size(), cudaMemcpyHostToDevice));
    *dst = static_cast<const double*>(d);
    return CARMPC_OK;
}

}  // namespace

}  // namespace carmpc

using namespace carmpc;

extern "C" {

int carmpc_qp_checker_create(int n, int R, const double* h_H, const double* h_F, const double* h_G, const double* h_Gx,
                             const double* h_Gc, const double* h_lo, const double* h_hi, const double* h_lb,
                             const double* h_ub, void** handle) {
    CARMPC_REQUIRE(handle != nullptr, "handle");
    CARMPC_REQUIRE(n >= 1 && n <= kCheckMaxN, "n must be in [1, 160]");
    CARMPC_REQUIRE(R >= 0 && R <= kCheckMaxR, "R must be in [0, 16000]");
    CARMPC_REQUIRE(h_H && h_F && h_lb && h_ub, "null matrix pointer");
    CARMPC_REQUIRE(R == 0 || (h_G && h_Gx && h_lo && h_hi), "null constraint pointer");
    for (size_t e = 0; e < (size_t)n * n; ++e) CARMPC_REQUIRE(isfinite(h_H[e]), "H must be finite");
    for (size_t e = 0; e < (size_t)n * 4; ++e) CARMPC_REQUIRE(isfinite(h_F[e]), "F must be finite");
    for (size_t e = 0; e < (size_t)R * n; ++e) CARMPC_REQUIRE(isfinite(h_G[e]), "G must be finite");
    for (size_t e = 0; e < (size_t)R * 4; ++e) CARMPC_REQUIRE(isfinite(h_Gx[e]), "Gx must be finite");
    for (int i = 0; i < R; ++i) {
        CARMPC_REQUIRE(!isnan(h_lo[i]) && !isnan(h_hi[i]) && h_lo[i] != INFINITY && h_hi[i] != -INFINITY, "row bounds");
        CARMPC_REQUIRE(h_Gc == nullptr || isfinite(h_Gc[i]), "Gc must be finite");
    }
    for (int j = 0; j < n; ++j)
        CARMPC_REQUIRE(!isnan(h_lb[j]) && !isnan(h_ub[j]) && h_lb[j] != INFINITY && h_ub[j] != -INFINITY, "box bounds");
    QPCheckHandle* q = new QPCheckHandle();
    q->kind = kQPCheck;
    CheckTables& t = q->t;
    t.n = n; t.R = R;
    int n_dev = 0;
    if (cudaGetDeviceCount(&n_dev) != cudaSuccess || n_dev == 0) {
        cudaGetLastError();
        q->host_only = true;
        *handle = q;
        return CARMPC_OK;
    }
    cudaGetDevice(&q->device);
    std::vector<double> H(h_H, h_H + (size_t)n * n), F(h_F, h_F + (size_t)n * 4), G, GT((size_t)n * R), Gx, Gc, lo, hi;
    if (R > 0) {
        G.assign(h_G, h_G + (size_t)R * n); Gx.assign(h_Gx, h_Gx + (size_t)R * 4);
        lo.assign(h_lo, h_lo + R); hi.assign(h_hi, h_hi + R);
        for (int i = 0; i < R; ++i)
            for (int j = 0; j < n; ++j) GT[(size_t)j * R + i] = G[(size_t)i * n + j];
    }
    std::vector<double> lb(h_lb, h_lb + n), ub(h_ub, h_ub + n);
    int rc = CARMPC_OK;
#define UPC(vec, field) do { rc = upload_doubles(q, vec, &t.field); if (rc != CARMPC_OK) { delete q; return rc; } } while (0)
    UPC(H, H); UPC(F, F); UPC(G, G); UPC(GT, GT); UPC(Gx, Gx); UPC(lo, lo); UPC(hi, hi); UPC(lb, lb); UPC(ub, ub);
    if (h_Gc && R > 0) { Gc.assign(h_Gc, h_Gc + R); UPC(Gc, Gc); } else t.Gc = nullptr;
#undef UPC
    t.gt_smem = sizeof(double) * (size_t)n * R <= kCheckSmemGT;
    *handle = q;
    return CARMPC_OK;
}

int carmpc_qp_check(void* checker, const double* d_x0, const double* h_xref, const double* d_c, int64_t batch,
                    const int32_t* d_status, const double* d_u_full, const double* d_cert, double* d_resid, void* stream) {
    QPCheckHandle* q = check_handle<QPCheckHandle>(checker, kQPCheck);
    CARMPC_REQUIRE(q != nullptr, "not a QP checker handle");
    CARMPC_REQUIRE(batch >= 0 && batch < (int64_t)1 << 31, "batch");
    CARMPC_REQUIRE(h_xref != nullptr, "h_xref");
    if (batch == 0) return CARMPC_OK;
    CARMPC_REQUIRE(d_x0 && d_status && d_u_full && d_cert && d_resid, "d_x0, d_status, d_u_full, d_cert and d_resid are required");
    for (int k = 0; k < 4; ++k) CARMPC_REQUIRE(isfinite(h_xref[k]), "h_xref must be finite");
    if (q->host_only) { set_error("carmpc_qp_check: this checker was created without a CUDA device"); return CARMPC_ERR_CUDA; }
    const CheckTables& t = q->t;
    CheckArgs a;
    memset(&a, 0, sizeof(a));
    a.x0 = d_x0; a.batch = batch; a.c = d_c;
    for (int k = 0; k < 4; ++k) a.xref[k] = h_xref[k];
    a.status = d_status; a.u_full = d_u_full; a.cert = d_cert; a.resid = d_resid;
    const size_t smem = sizeof(double) * ((t.gt_smem ? (size_t)t.n * t.R : 0) + (size_t)(kCheckThreads / 32) * t.n);
    int per_sm = 0;
    { const int rc = kernel_config(reinterpret_cast<const void*>(qp_check_kernel), kCheckThreads, smem, &per_sm); if (rc != CARMPC_OK) return rc; }
    const int64_t need = (batch + kCheckThreads / 32 - 1) / (kCheckThreads / 32);
    const int blocks = (int)std::max<int64_t>(1, std::min<int64_t>(need, (int64_t)sm_count() * std::max(per_sm, 1)));
    qp_check_kernel<<<blocks, kCheckThreads, smem, (cudaStream_t)stream>>>(t, a);
    CARMPC_CUDA(cudaGetLastError());
    return CARMPC_OK;
}

}  // extern "C"
