// Derivatives of certified QP solutions with respect to the initial state and the disturbance (carmpc_qp_sensitivity).
//
// A solved sample's certificate row y (carmpc_qp_solve d_cert) names its active rows S = {i : y_i != 0} among the m
// general and n box rows, A = [G; I].  On the critical region of S the solution is affine in p = (x0, c):
//       M lambda = AUu_S (x0 - xref) + Gx_S x0 + Gc_S c - b_S ,   u = Uu (x0 - xref) - AH_S' lambda ,   M = A_S H^-1 A_S'
// hence (box rows: Gx = Gc = 0)
//       dlam/dx0 = M^-1 (AUu_S + Gx_S)      dlam/dc = M^-1 Gc_S
//       du/dx0   = Uu - AH_S' dlam/dx0      du/dc   = -AH_S' dlam/dc
//       dV/dx0   = F'u + Gx_S' lambda       dV/dc   = Gc_S' lambda          (envelope theorem, V = the objective)
// with the shared PolishTables.  None of it depends on xref.  One warp per sample, as in the polish: gather M into packed
// shared memory, factor it with the polish's division-free Cholesky and pivot-skip rule, solve the five right-hand sides,
// and classify the sample (flags below).
//
// The factor and the solve are written again here rather than shared with polish_kernel: there they are lambdas over
// that kernel's shared-memory layout and its register budget is tuned; shared code would have to branch on its caller.
#include <math.h>

#include <algorithm>

#include "qp_internal.cuh"

namespace carmpc {

namespace {

constexpr int kSensThreads = 128;
constexpr int kSensWarps = kSensThreads / 32;
// The pivot rule of the polish's factorisation (qp_polish.cu): the diagonal is raised by kPivotReg of itself, and a pivot
// that falls to kPivotSkip of its original diagonal marks a row that depends on the earlier ones (its lambda is 0).
constexpr double kPivotReg = 1e-13;
constexpr double kPivotSkip = 1e-11;
// flags (carmpc.h)
constexpr int kFlagDerivative = 1, kFlagWeak = 2, kFlagDependent = 4, kFlagTooMany = 8;

__device__ __forceinline__ int tri(int i, int j) { return i * (i + 1) / 2 + j; }     // j <= i

__device__ __forceinline__ double warp_max(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

struct SensArgs {
    const double* x0; int stride; const double* cdist;
    const int32_t* status; const double* u_full; const double* cert;
    int rows; double* jac; double* grad; int32_t* flags;
    const double* Px; const double* Pc; const double* pre_lo; const double* pre_hi;
    int na_cap;
};

// per warp: M packed (na_cap (na_cap + 1) / 2), diag0 / reciprocal pivots (na_cap), right-hand sides (5 na_cap), lambda
// (na_cap), u (n) as doubles, then the active rows (na_cap ints)
__host__ __device__ inline size_t sens_per_warp(int n, int na_cap) {
    const size_t d = (size_t)na_cap * (na_cap + 1) / 2 + 7 * (size_t)na_cap + n;
    return (d * sizeof(double) + sizeof(int) * (size_t)na_cap + 15) & ~size_t(15);
}

// Cholesky of the packed lower triangle M (na x na) in place; diag0 holds the original diagonal on entry and 1 / L_jj on
// exit (0 for a skipped pivot, whose column of L is zeroed).  Returns the number of skipped pivots.  Same arithmetic as
// the polish.
__device__ int factor_packed(double* M, double* diag0, int na, int lane) {
    int skipped = 0;
    for (int j = 0; j < na; ++j) {
        const double d = M[tri(j, 0) + j];
        const bool skip = !(d > kPivotSkip * diag0[j]);
        const double rinv = skip ? 0.0 : rsqrt(d);
        skipped += skip ? 1 : 0;
        __syncwarp();
        if (lane == 0) diag0[j] = rinv;
        for (int i = j + 1 + lane; i < na; i += 32) M[tri(i, 0) + j] *= rinv;
        __syncwarp();
        if (!skip) {
            const int li = lane >> 2, lk = lane & 3;                  // lanes as an 8 x 4 grid over (i, k), j < k <= i
            for (int i = j + 1 + li; i < na; i += 8) {
                const int ti = tri(i, 0);
                const double lij = M[ti + j];
                for (int k = j + 1 + lk; k <= i; k += 4) M[ti + k] -= lij * M[tri(k, 0) + j];
            }
        }
        __syncwarp();
    }
    return skipped;
}

// L L' X = R for the five columns of R ([na][5]) in place
__device__ void solve5_packed(const double* M, const double* rinv, double* R, int na, int lane) {
    for (int j = 0; j < na; ++j) {
        double y[5];
#pragma unroll
        for (int c = 0; c < 5; ++c) y[c] = R[j * 5 + c] * rinv[j];
        __syncwarp();
        if (lane == 0)
#pragma unroll
            for (int c = 0; c < 5; ++c) R[j * 5 + c] = y[c];
        for (int i = j + 1 + lane; i < na; i += 32) {
            const double l = M[tri(i, 0) + j];
#pragma unroll
            for (int c = 0; c < 5; ++c) R[i * 5 + c] -= l * y[c];
        }
        __syncwarp();
    }
    for (int j = na - 1; j >= 0; --j) {
        double x[5];
#pragma unroll
        for (int c = 0; c < 5; ++c) x[c] = R[j * 5 + c] * rinv[j];
        const int tj = tri(j, 0);
        __syncwarp();
        if (lane == 0)
#pragma unroll
            for (int c = 0; c < 5; ++c) R[j * 5 + c] = x[c];
        for (int i = lane; i < j; i += 32) {
            const double l = M[tj + i];
#pragma unroll
            for (int c = 0; c < 5; ++c) R[i * 5 + c] -= l * x[c];
        }
        __syncwarp();
    }
}

__global__ void __launch_bounds__(kSensThreads) sensitivity_kernel(const PolishTables T, const SensArgs A, int batch) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int n = T.n, m = T.m, mt = T.mt, width = T.mt + T.kpre, cap = A.na_cap;
    unsigned char* base = smem_raw + (size_t)warp * sens_per_warp(n, cap);
    double* M = reinterpret_cast<double*>(base);
    double* diag0 = M + (size_t)cap * (cap + 1) / 2;
    double* R = diag0 + cap;
    double* lam = R + 5 * cap;
    double* u = lam + cap;
    int* act = reinterpret_cast<int*>(u + n);
    const double NaN = __longlong_as_double(0x7ff8000000000000ll);

    for (int s = blockIdx.x * kSensWarps + warp; s < batch; s += gridDim.x * kSensWarps) {
        double* jac = A.jac ? A.jac + (size_t)s * A.rows * 5 : nullptr;
        if (A.status[s] != CARMPC_QP_SOLVED) {
            if (jac) for (int e = lane; e < A.rows * 5; e += 32) jac[e] = NaN;
            if (A.grad && lane < 5) A.grad[(size_t)s * 5 + lane] = NaN;
            if (lane == 0) A.flags[s] = 0;
            continue;
        }
        double x0[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) x0[k] = A.x0[(size_t)k * A.stride + s];
        const double cd = A.cdist ? A.cdist[s] : 0.0;
        const double* y = A.cert + (size_t)s * width;
        // ---- S in row order, lambda in the handle's orientation, and the multiplier part of dV ----
        double g[5] = {0, 0, 0, 0, 0};
        double lmax = 0.0;
        int na = 0;
        for (int i0 = 0; i0 < mt; i0 += 32) {
            const int i = i0 + lane;
            const double yi = i < mt ? y[i] : 0.0;
            const bool on = yi != 0.0;
            const unsigned mask = __ballot_sync(0xffffffffu, on);
            if (on) {
                const double l = i < m ? T.rsign[i] * yi : yi;
                const int p = na + __popc(mask & ((1u << lane) - 1u));
                if (p < cap) { act[p] = i; lam[p] = l; }
                lmax = fmax(lmax, fabs(l));
                if (i < m) {
                    const double* gx = T.Gx + (size_t)i * 4;
#pragma unroll
                    for (int k = 0; k < 4; ++k) g[k] += gx[k] * l;
                    g[4] += T.Gc[i] * l;
                }
            }
            na += __popc(mask);
        }
        lmax = warp_max(lmax);
        // ---- u and the F'u part of dV ----
        for (int j = lane; j < n; j += 32) {
            const double uj = A.u_full[(size_t)s * n + j];
            u[j] = uj;
            const double* f = T.F + (size_t)j * 4;
#pragma unroll
            for (int k = 0; k < 4; ++k) g[k] += f[k] * uj;
        }
#pragma unroll
        for (int k = 0; k < 5; ++k) g[k] = warp_sum(g[k]);
        if (A.grad && lane == 0)
#pragma unroll
            for (int k = 0; k < 5; ++k) A.grad[(size_t)s * 5 + k] = g[k];
        if (na > cap) {                                   // no solver certificate has that many rows
            if (jac) for (int e = lane; e < A.rows * 5; e += 32) jac[e] = NaN;
            if (lane == 0) A.flags[s] = kFlagTooMany;
            continue;
        }
        __syncwarp();
        // ---- weak multipliers on S ----
        bool weak = false;
        for (int a = lane; a < na; a += 32) weak = weak || !(fabs(lam[a]) > kSignTol * (1.0 + lmax));
        // ---- rows outside S at a bound: A u is evaluated from u (the table form AUu (x0 - xref) + ... would need xref) ----
        for (int i = lane; i < mt; i += 32) {
            if (y[i] != 0.0) continue;
            double t;
            if (i < m) {
                const double* gi = T.G + (size_t)i * n;
                const double* gx = T.Gx + (size_t)i * 4;
                t = gx[0] * x0[0] + gx[1] * x0[1] + gx[2] * x0[2] + gx[3] * x0[3] + T.Gc[i] * cd;
                for (int j = 0; j < n; ++j) t += gi[j] * u[j];
            } else {
                t = u[i - m];
            }
            weak = weak || t >= T.hi[i] - kFeasTol || t <= T.lo[i] + kFeasTol;
        }
        for (int k = lane; k < T.kpre; k += 32) {
            const double v = A.Px[k * 4 + 0] * x0[0] + A.Px[k * 4 + 1] * x0[1] + A.Px[k * 4 + 2] * x0[2] +
                             A.Px[k * 4 + 3] * x0[3] + A.Pc[k] * cd;
            weak = weak || v >= A.pre_hi[k] - kFeasTol || v <= A.pre_lo[k] + kFeasTol;
        }
        weak = __any_sync(0xffffffffu, weak);
        // ---- M = AHA[S, S] (lower triangle), right-hand sides [AUu_S + Gx_S | Gc_S] ----
        for (int e = lane; e < na * (na + 1) / 2; e += 32) {
            int a = (int)((sqrt(8.0 * e + 1.0) - 1.0) * 0.5);
            while (tri(a + 1, 0) <= e) ++a;
            while (tri(a, 0) > e) --a;
            const int b = e - tri(a, 0);
            double v = T.AHA[(size_t)act[a] * mt + act[b]];
            if (a == b) { diag0[a] = v; v += kPivotReg * v; }
            M[e] = v;
        }
        for (int a = lane; a < na; a += 32) {
            const int i = act[a];
            const double* w = T.AUu + (size_t)i * 4;
#pragma unroll
            for (int k = 0; k < 4; ++k) R[a * 5 + k] = w[k] + (i < m ? T.Gx[(size_t)i * 4 + k] : 0.0);
            R[a * 5 + 4] = i < m ? T.Gc[i] : 0.0;
        }
        __syncwarp();
        const int skipped = factor_packed(M, diag0, na, lane);
        solve5_packed(M, diag0, R, na, lane);
        // ---- du/d(x0, c) of the leading rows variables ----
        if (jac) {
            for (int r = lane; r < A.rows; r += 32) {
                double acc[5];
                const double* w = T.Uu + (size_t)r * 4;
#pragma unroll
                for (int k = 0; k < 4; ++k) acc[k] = w[k];
                acc[4] = 0.0;
                for (int a = 0; a < na; ++a) {
                    const double h = T.AH[(size_t)act[a] * n + r];
#pragma unroll
                    for (int k = 0; k < 5; ++k) acc[k] -= h * R[a * 5 + k];
                }
#pragma unroll
                for (int k = 0; k < 5; ++k) jac[(size_t)r * 5 + k] = acc[k];
            }
        }
        if (lane == 0) A.flags[s] = (weak ? kFlagWeak : 0) | (skipped ? kFlagDependent : 0) |
                                    (!weak && !skipped ? kFlagDerivative : 0);
        __syncwarp();
    }
}

}  // namespace

int sensitivity_launch(QPHandle* qh, const double* d_x0, const double* d_c, int64_t batch, const int32_t* d_status,
                       const double* d_u_full, const double* d_cert, int rows, double* d_jac, double* d_grad,
                       int32_t* d_flags, cudaStream_t st) {
    if (batch <= 0) return CARMPC_OK;
    SensArgs a = {};
    a.x0 = d_x0; a.stride = (int)batch; a.cdist = d_c; a.status = d_status; a.u_full = d_u_full; a.cert = d_cert;
    a.rows = rows; a.jac = d_jac; a.grad = d_grad; a.flags = d_flags;
    a.Px = qh->admm.Px; a.Pc = qh->admm.Pc; a.pre_lo = qh->admm.pre_lo; a.pre_hi = qh->admm.pre_hi;
    a.na_cap = std::min(kPolishMaxActive, qh->polish.mt);
    const size_t smem = sens_per_warp(qh->polish.n, a.na_cap) * kSensWarps;
    int per_sm = 0;
    { const int rc = kernel_config(reinterpret_cast<const void*>(sensitivity_kernel), kSensThreads, smem, &per_sm); if (rc != CARMPC_OK) return rc; }
    const int blocks = (int)std::max<int64_t>(1, std::min<int64_t>((batch + kSensWarps - 1) / kSensWarps, (int64_t)qh->sm * per_sm));
    sensitivity_kernel<<<blocks, kSensThreads, smem, st>>>(qh->polish, a, (int)batch);
    CARMPC_CUDA(cudaGetLastError());
    return CARMPC_OK;
}

}  // namespace carmpc
