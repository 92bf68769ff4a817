// Float64 active-set polish of the batched QP (second kernel of a pass; see qp_internal.cuh).
//
// Given the active-set guess of the float32 ADMM (sign per constraint row: +1 at its upper bound, -1 at its lower), one
// warp per sample solves the equality-constrained QP exactly through the Schur complement on the shared matrices
//       u = u_unc - (A H^-1)'_act lambda ,   (A_act H^-1 A_act' + delta I) lambda = A_act u_unc - b_act ,   u_unc = -H^-1 q
// then checks the KKT conditions in float64 (every row within its bounds, multiplier signs right).  A wrong guess is
// repaired (drop rows with a wrong-signed multiplier, add the most violated row) a few times.  What leaves this kernel
// with status 0 and polished = 1 is a certified optimum of the reference's QP (lib/mpc.py:321-332) to ~1e-10.
#include <math.h>

#include <algorithm>

#include "qp_internal.cuh"

namespace carmpc {

namespace {

constexpr int kPolishRounds = 10;
constexpr int kPolishSmallActive = 32;
constexpr int kAddPerRound = 3;      // violated rows added to the active set per repair round
constexpr int kPolishThreads = 128;

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ double warp_max(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

struct PolishSmemLayout {
    int na_max;
    size_t per_warp;
};

__host__ __device__ inline PolishSmemLayout polish_layout(int n, int mt, int na_cap) {
    PolishSmemLayout L;
    L.na_max = na_cap;
    if (L.na_max > mt) L.na_max = mt;
    if (L.na_max < 1) L.na_max = 1;
    size_t d = 0;
    d += 2 * (size_t)n;                                      // u_unc, u
    d += (size_t)mt;                                         // t = A u_unc + bound shift
    d += (size_t)L.na_max * (L.na_max + 1) / 2;              // M, packed lower triangle
    d += 3 * (size_t)L.na_max;                               // rhs / lambda, b, diag0
    size_t bytes = d * sizeof(double);
    bytes += sizeof(int) * (size_t)L.na_max;                 // act
    bytes += sizeof(int) * 16;                               // rows added by the repair, newest first
    bytes += (size_t)((mt + 15) & ~15);                      // sgn
    L.per_warp = (bytes + 15) & ~size_t(15);
    return L;
}

__device__ __forceinline__ int tri(int i, int j) { return i * (i + 1) / 2 + j; }     // j <= i

// Table gathers of the u update / KKT check: the tables (A H^-1, A H^-1 A') live in L2, so what these loops wait for is load
// latency.  Volatile asm keeps the loads of a batch together in front of the multiply-adds that consume them (left to
// itself ptxas interleaves load -> DFMA -> load through one register pair, one L2 round trip after the other).
__device__ __forceinline__ double ldg_table(const double* p) {
    double v;
    asm volatile("ld.global.nc.f64 %0, [%1];" : "=d"(v) : "l"(p));
    return v;
}

// (A u_unc)_i = AUu_i . dx
__device__ __forceinline__ double T_auu(const PolishTables& T, int i, const double (&dx)[4]) {
    const double* w = T.AUu + (size_t)i * 4;
    return w[0] * dx[0] + w[1] * dx[1] + w[2] * dx[2] + w[3] * dx[3];
}

// 7 CTAs of 4 warps per SM (72 registers, 28.6 KB of shared memory each): measured against 3..10 CTAs per SM with the
// matching register budgets, fewer warps with more registers (deeper load batching) is slower, more warps no faster.
// One instantiation per mode, so that the cold launch (10^6 samples) carries none of the seed / record / certificate /
// pre-check code (round 1: one kernel for all modes, 6,100 SASS instructions, instruction-fetch stalls in the cold launch):
//   SEEDED   followers of a seeded map (active set and records of an anchor),   PRECHECK  u-independent rows / finiteness
//   (active-set reuse: closed loop and followers),   RECWRITE  anchors exporting their multiplier map.
template <bool SEEDED, bool PRECHECK, bool RECWRITE>
__global__ void __launch_bounds__(kPolishThreads, 7) polish_kernel(const PolishTables T, const PolishBatch B) {
    const int* const b_seed = SEEDED ? B.seed : nullptr;
    const bool b_precheck = PRECHECK && B.precheck != 0;
    const bool b_rec_read = SEEDED && B.rec_read != 0;
    const bool b_rec_write = RECWRITE && B.rec_write != 0;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    constexpr int warps_per_cta = kPolishThreads / 32;
    const int n = T.n, m = T.m, mt = T.mt;
    const PolishSmemLayout L = polish_layout(n, mt, B.na_cap);
    unsigned char* base = smem_raw + (size_t)warp * L.per_warp;
    double* uunc = reinterpret_cast<double*>(base);
    double* u = uunc + n;
    double* tsh = u + n;                 // t_i = (A u_unc)_i + Gx_i x0 + Gc_i c: row i is within bounds iff lo_i <= t_i - corr_i <= hi_i
    double* M = tsh + mt;
    double* rhs = M + (size_t)L.na_max * (L.na_max + 1) / 2;
    double* bact = rhs + L.na_max;
    double* diag0 = bact + L.na_max;
    int* act = reinterpret_cast<int*>(diag0 + L.na_max);
    int* added = act + L.na_max;
    signed char* sgn = reinterpret_cast<signed char*>(added + 16);
    const double NaN = __longlong_as_double(0x7ff8000000000000ll);

    const int gw = blockIdx.x * warps_per_cta + warp, nw = gridDim.x * warps_per_cta;
    const int count = B.count_dev ? min(*B.count_dev, B.count) : B.count;
    for (int qi = gw; qi < count; qi += nw) {
        const int sample = B.idx_list ? B.idx_list[qi] : qi;
        const int st_in = B.status[sample];
        __syncwarp();
        if (st_in == CARMPC_QP_INFEASIBLE) {
            if (lane == 0) {
                if (B.u0) { B.u0[sample] = NaN; B.u0[B.stride + sample] = NaN; }
                if (B.objective) B.objective[sample] = INFINITY;
                if (B.polished) B.polished[sample] = 0;
            }
            if (B.u_full) for (int j = lane; j < n; j += 32) B.u_full[(size_t)sample * n + j] = NaN;
            continue;
        }
        double x0[4], dx[4];
#pragma unroll
        for (int c = 0; c < 4; ++c) { x0[c] = B.x0[(size_t)c * B.stride + sample]; dx[c] = x0[c] - B.xref[c]; }
        const double cd = B.cdist ? B.cdist[sample] : 0.0;
        // seeded: the guess is the certified set of the sample's anchor (nothing to try when the anchor was infeasible)
        const int sign_src = b_seed ? b_seed[sample] : sample;
        const bool seed_ok = !b_seed || B.status[sign_src] == CARMPC_QP_SOLVED;
        // everything unconstrained is linear in dx:  u_unc = -H^-1 F dx = Uu dx ,  A u_unc = (A Uu) dx
        for (int j = lane; j < n; j += 32) {
            const double* w = T.Uu + (size_t)j * 4;
            uunc[j] = w[0] * dx[0] + w[1] * dx[1] + w[2] * dx[2] + w[3] * dx[3];
        }
        for (int i = lane; i < mt; i += 32) {
            const double* w = T.AUu + (size_t)i * 4;
            double t = w[0] * dx[0] + w[1] * dx[1] + w[2] * dx[2] + w[3] * dx[3];
            if (i < m) {
                const double* gx = T.Gx + (size_t)i * 4;
                t += gx[0] * x0[0] + gx[1] * x0[1] + gx[2] * x0[2] + gx[3] * x0[3] + T.Gc[i] * cd;
            }
            tsh[i] = t;
            sgn[i] = B.sign[(size_t)sign_src * mt + i];
        }
        int n_added = 0;
        __syncwarp();

        bool certified = false, overflow = false;
        int na = 0;
        int max_rounds = B.rounds < 0 ? kPolishRounds : B.rounds;
        if (b_precheck) {
            // what the ADMM slot refill checks before it starts a sample: finite state, rows that do not depend on u
            bool pre_ok = isfinite(x0[0]) && isfinite(x0[1]) && isfinite(x0[2]) && isfinite(x0[3]);
            for (int k = 0; k < B.kpre; ++k) {
                const double v = B.Px[k * 4 + 0] * x0[0] + B.Px[k * 4 + 1] * x0[1] + B.Px[k * 4 + 2] * x0[2] +
                                 B.Px[k * 4 + 3] * x0[3] + B.Pc[k] * cd;
                pre_ok = pre_ok && v <= B.pre_hi[k] && v >= B.pre_lo[k];
            }
            if (!pre_ok || !seed_ok) max_rounds = 0;                       // not certified: the ADMM pass decides
            // Seeded map: a violated u-independent row is infeasibility by itself; an infeasible anchor may have exported a
            // Farkas certificate y (A'y = 0 exactly, box rows absorb the residual), whose support value is affine in x0:
            // S(x0) = c0 - cx.x0 < 0 proves that THIS state is infeasible as well.
            bool proven_infeasible = b_seed != nullptr && !pre_ok;
            if (b_seed && b_rec_read && pre_ok && B.status[sign_src] == CARMPC_QP_INFEASIBLE) {
                const int rec = B.rec_of[sign_src];
                if (rec >= 0 && B.rec_act[(size_t)rec * (kPolishSmallActive + 1)] == -2) {
                    const double* r = B.rec_lam + (size_t)rec * kPolishSmallActive * 5;
                    const double S = r[4] - (r[0] * x0[0] + r[1] * x0[1] + r[2] * x0[2] + r[3] * x0[3]);
                    const double margin = 1e-9 * (r[9] + r[5] * fabs(x0[0]) + r[6] * fabs(x0[1]) + r[7] * fabs(x0[2]) + r[8] * fabs(x0[3]));
                    proven_infeasible = S < -margin;
                }
            }
            if (proven_infeasible) {
                if (B.cert) {
                    // the anchor's exported row is the certificate its record holds (farkas_kernel mode 0 wrote it)
                    double* row = B.cert + (size_t)sample * (mt + T.kpre);
                    if (!pre_ok) store_pre_certificate(row, mt, T.kpre, B.Px, B.Pc, B.pre_lo, B.pre_hi, x0, cd, lane);
                    else for (int e = lane; e < mt + T.kpre; e += 32) row[e] = B.cert[(size_t)sign_src * (mt + T.kpre) + e];
                }
                if (lane == 0) {
                    B.status[sample] = CARMPC_QP_INFEASIBLE;
                    if (B.iters_out) B.iters_out[sample] = 0;
                    if (B.u0) { B.u0[sample] = NaN; B.u0[B.stride + sample] = NaN; }
                    if (B.objective) B.objective[sample] = INFINITY;
                    if (B.polished) B.polished[sample] = 0;
                    if (B.stats) atomicAdd(B.stats + 13, 1ull);
                }
                if (B.u_full) for (int j = lane; j < n; j += 32) B.u_full[(size_t)sample * n + j] = NaN;
                continue;
            }
        }
        // L y = rhs, L' x = y in place (M holds the factor, diag0 the reciprocal pivots; skipped pivots give 0)
        auto solve_in_place = [&]() {
            for (int j = 0; j < na; ++j) {
                const double y = rhs[j] * diag0[j];
                __syncwarp();
                if (lane == 0) rhs[j] = y;
                for (int i = j + 1 + lane; i < na; i += 32) rhs[i] -= M[tri(i, 0) + j] * y;
                __syncwarp();
            }
            for (int j = na - 1; j >= 0; --j) {
                const double x = rhs[j] * diag0[j];
                const int tj = tri(j, 0);
                __syncwarp();
                if (lane == 0) rhs[j] = x;
                for (int i = lane; i < j; i += 32) rhs[i] -= M[tj + i] * x;
                __syncwarp();
            }
        };
        // Seeded from an anchor that exported its multiplier map: on the anchor's critical region lambda is affine in x0
        // (explicit-MPC form), so round 0 needs no factorisation - only the KKT certificate below decides.
        bool lam_ready = false;
        if (b_rec_read && b_seed && seed_ok && max_rounds > 0 && B.cdist == nullptr) {
            const int rec = B.rec_of[sign_src];
            if (rec >= 0) {
                const int* ra = B.rec_act + (size_t)rec * (kPolishSmallActive + 1);
                const int rna = ra[0];
                if (rna >= 0 && rna <= L.na_max) {
                    na = rna;
                    for (int a = lane; a < na; a += 32) {
                        const int i = ra[1 + a];
                        const double* lr = B.rec_lam + ((size_t)rec * kPolishSmallActive + a) * 5;
                        act[a] = i;
                        rhs[a] = lr[0] * x0[0] + lr[1] * x0[1] + lr[2] * x0[2] + lr[3] * x0[3] + lr[4];
                        bact[a] = (sgn[i] > 0 ? T.hi[i] : T.lo[i]) - (tsh[i] - T_auu(T, i, dx));
                    }
                    lam_ready = true;
                    __syncwarp();
                }
            }
        }
        int rounds_used = 0;
        for (int round = 0; round < max_rounds && !certified; ++round) {
            rounds_used = round;
            if (!(round == 0 && lam_ready)) {
            // ---- active list: rows added by the repair first (newest first: they keep their pivot when the set is
            //      linearly dependent, and an older guess gets the zero multiplier), then the ADMM guess by index ----
            na = 0;
            for (int a = 0; a < n_added; ++a) {
                const int i = added[a];
                if (sgn[i] != 0) { if (lane == 0 && na < L.na_max) act[na] = i; ++na; }
            }
            for (int i0 = 0; i0 < mt; i0 += 32) {
                const int i = i0 + lane;
                bool on = i < mt && sgn[i] != 0;
                if (on) for (int a = 0; a < n_added; ++a) on = on && added[a] != i;
                const unsigned mask = __ballot_sync(0xffffffffu, on);
                const int p = na + __popc(mask & ((1u << lane) - 1u));
                if (on && p < L.na_max) act[p] = i;
                na += __popc(mask);
            }
            if (na > L.na_max) { overflow = true; break; }
            __syncwarp();
            // ---- M = AHA[act, act] (lower triangle), rhs = A_act u_unc - b_act ----
            for (int e = lane; e < na * (na + 1) / 2; e += 32) {
                int a = (int)((sqrt(8.0 * e + 1.0) - 1.0) * 0.5);
                while (tri(a + 1, 0) <= e) ++a;
                while (tri(a, 0) > e) --a;
                const int b = e - tri(a, 0);
                double v = T.AHA[(size_t)act[a] * mt + act[b]];
                if (a == b) { diag0[a] = v; v += 1e-13 * v; }
                M[e] = v;
            }
            for (int a = lane; a < na; a += 32) {
                const int i = act[a];
                const double bound = sgn[i] > 0 ? T.hi[i] : T.lo[i];
                bact[a] = bound - (tsh[i] - T_auu(T, i, dx));          // bound on A u: hi - shift
                rhs[a] = tsh[i] - bound;
            }
            __syncwarp();
            // ---- Cholesky with pivot skipping (a row that depends on earlier ones gets lambda = 0).  diag0[j] is
            //      overwritten by 1 / L_jj (0 for a skipped pivot) so that the solves below are division-free ----
            for (int j = 0; j < na; ++j) {
                const int tj = tri(j, 0);
                const double d = M[tj + j];
                const bool skip = !(d > 1e-11 * diag0[j]);
                const double rinv = skip ? 0.0 : rsqrt(d);                // every lane computes the same value
                __syncwarp();
                if (lane == 0) diag0[j] = rinv;
                for (int i = j + 1 + lane; i < na; i += 32) M[tri(i, 0) + j] *= rinv;      // L_ij (0 when skipped)
                __syncwarp();
                if (!skip) {
                    // trailing update M[i][k] -= L_ij L_kj over the triangle j < k <= i, lanes as an 8 x 4 grid of (i, k)
                    const int li = lane >> 2, lk = lane & 3;
                    for (int i = j + 1 + li; i < na; i += 8) {
                        const int ti = tri(i, 0);
                        const double lij = M[ti + j];
                        int k = j + 1 + lk;
                        // four independent (load, load, fma, store) chains per pass: with many active rows this loop is
                        // a chain of shared-memory round trips otherwise (no lane writes what another one reads here)
                        for (; k + 12 <= i; k += 16) {
                            const double c0 = M[tri(k, 0) + j], c1 = M[tri(k + 4, 0) + j], c2 = M[tri(k + 8, 0) + j], c3 = M[tri(k + 12, 0) + j];
                            const double m0 = M[ti + k], m1 = M[ti + k + 4], m2 = M[ti + k + 8], m3 = M[ti + k + 12];
                            M[ti + k] = m0 - lij * c0; M[ti + k + 4] = m1 - lij * c1;
                            M[ti + k + 8] = m2 - lij * c2; M[ti + k + 12] = m3 - lij * c3;
                        }
                        for (; k <= i; k += 4) M[ti + k] -= lij * M[tri(k, 0) + j];
                    }
                }
                __syncwarp();
            }
            solve_in_place();
            }
            // rhs now holds lambda (signed: positive pushes against an upper bound)
            // ---- u = u_unc - (AH)'_act lambda : kUChunk variables per lane at a time, so that every active row contributes
            //      kUChunk independent loads (the tables live in L2: latency, not bandwidth, is what this loop waits for) ----
            constexpr int kUChunk = 2, kRowChunk = 5;
            for (int j0 = 0; j0 < n; j0 += 32 * kUChunk) {
                double acc[kUChunk];
                int jj[kUChunk];
#pragma unroll
                for (int c = 0; c < kUChunk; ++c) { jj[c] = j0 + 32 * c + lane; acc[c] = jj[c] < n ? uunc[jj[c]] : 0.0; if (jj[c] >= n) jj[c] = 0; }
                int a = 0;
                for (; a + 4 <= na; a += 4) {                         // 4 active rows x kUChunk loads in flight
                    double v[4][kUChunk], la[4];
#pragma unroll
                    for (int r = 0; r < 4; ++r) {
                        la[r] = rhs[a + r];
                        const double* row = T.AH + (size_t)act[a + r] * n;
#pragma unroll
                        for (int c = 0; c < kUChunk; ++c) v[r][c] = ldg_table(row + jj[c]);
                    }
#pragma unroll
                    for (int r = 0; r < 4; ++r)
#pragma unroll
                        for (int c = 0; c < kUChunk; ++c) acc[c] -= v[r][c] * la[r];
                }
                for (; a < na; ++a) {
                    const double la = rhs[a];
                    const double* row = T.AH + (size_t)act[a] * n;
                    double v[kUChunk];
#pragma unroll
                    for (int c = 0; c < kUChunk; ++c) v[c] = ldg_table(row + jj[c]);
#pragma unroll
                    for (int c = 0; c < kUChunk; ++c) acc[c] -= v[c] * la;
                }
#pragma unroll
                for (int c = 0; c < kUChunk; ++c) if (j0 + 32 * c + lane < n) u[j0 + 32 * c + lane] = acc[c];
            }
            // ---- KKT check: every row within its bounds, multiplier signs right (kRowChunk rows per lane at a time) ----
            double worst = 0.0;
            int worst_i = -1, worst_sign = 0;
            for (int i0 = 0; i0 < mt; i0 += 32 * kRowChunk) {
                double acc[kRowChunk];
                int ii[kRowChunk];
#pragma unroll
                for (int c = 0; c < kRowChunk; ++c) { ii[c] = i0 + 32 * c + lane; acc[c] = ii[c] < mt ? tsh[ii[c]] : 0.0; if (ii[c] >= mt) ii[c] = 0; }
                int a = 0;
                for (; a + 2 <= na; a += 2) {                         // 2 active rows x kRowChunk loads in flight
                    double v[2][kRowChunk], la[2];
#pragma unroll
                    for (int r = 0; r < 2; ++r) {
                        la[r] = rhs[a + r];
                        const double* row = T.AHA + (size_t)act[a + r] * mt;
#pragma unroll
                        for (int c = 0; c < kRowChunk; ++c) v[r][c] = ldg_table(row + ii[c]);
                    }
#pragma unroll
                    for (int r = 0; r < 2; ++r)
#pragma unroll
                        for (int c = 0; c < kRowChunk; ++c) acc[c] -= v[r][c] * la[r];
                }
                for (; a < na; ++a) {
                    const double la = rhs[a];
                    const double* row = T.AHA + (size_t)act[a] * mt;
                    double v[kRowChunk];
#pragma unroll
                    for (int c = 0; c < kRowChunk; ++c) v[c] = ldg_table(row + ii[c]);
#pragma unroll
                    for (int c = 0; c < kRowChunk; ++c) acc[c] -= v[c] * la;
                }
#pragma unroll
                for (int c = 0; c < kRowChunk; ++c) {
                    const int i = i0 + 32 * c + lane;
                    if (i >= mt) continue;
                    const double h = T.hi[i], l = T.lo[i];
                    if (isinf(h) && isinf(l)) continue;
                    const double vu = acc[c] - h, vl = l - acc[c];
                    const double v = fmax(vu, vl);
                    if (v > worst) { worst = v; worst_i = i; worst_sign = vu >= vl ? 1 : -1; }
                }
            }
            // the (up to) kAddPerRound most violated rows, one per lane
            int n_add = 0, add_is[kAddPerRound], add_sg[kAddPerRound];
            {
                double wv = worst_i >= 0 ? worst : -1.0;
#pragma unroll
                for (int t = 0; t < kAddPerRound; ++t) {
                    const double wmax = warp_max(wv);
                    if (!(wmax > kFeasTol)) break;                         // uniform
                    const unsigned who = __ballot_sync(0xffffffffu, wv == wmax);
                    const int src = __ffs(who) - 1;
                    add_is[n_add] = __shfl_sync(0xffffffffu, worst_i, src);
                    add_sg[n_add] = __shfl_sync(0xffffffffu, worst_sign, src);
                    ++n_add;
                    if (lane == src) wv = -1.0;
                }
            }
            double lam_max = 0.0;
            for (int a = lane; a < na; a += 32) lam_max = fmax(lam_max, fabs(rhs[a]));
            lam_max = warp_max(lam_max);
            int n_bad = 0;
            for (int a = lane; a < na; a += 32) {
                const int i = act[a];
                if (rhs[a] * (double)sgn[i] < -kSignTol * (1.0 + lam_max)) { sgn[i] = 0; ++n_bad; }
            }
            n_bad = __reduce_add_sync(0xffffffffu, n_bad);
            __syncwarp();
            if (n_add == 0 && n_bad == 0) { certified = true; break; }
            for (int t = n_add - 1; t >= 0; --t) {                         // the most violated row ends up first
                const int add_i = add_is[t];
                int k = 0;
                for (int a = 0; a < n_added; ++a) if (added[a] != add_i) ++k;
                __syncwarp();
                if (lane == 0) {
                    sgn[add_i] = (signed char)add_sg[t];
                    int w = 0;                                         // move / insert add_i at the front
                    for (int a = 0; a < n_added; ++a) if (added[a] != add_i) added[w++] = added[a];
                    const int keep = w < 15 ? w : 15;
                    for (int a = keep; a > 0; --a) added[a] = added[a - 1];
                    added[0] = add_i;
                }
                n_added = (k < 15 ? k : 15) + 1;
                __syncwarp();
            }
            __syncwarp();
        }

        if (B.stats && lane == 0 && !(overflow && !certified && B.overflow_list != nullptr)) {
            atomicAdd(B.stats + (certified ? (rounds_used < 9 ? rounds_used : 9) : 10), 1ull);
            if (lam_ready) atomicAdd(B.stats + 11, 1ull);
            if (lam_ready && certified && rounds_used == 0) atomicAdd(B.stats + 12, 1ull);
        }
        double obj;
        if (!certified && overflow && B.overflow_list != nullptr) {
            // more active rows than this launch's shared-memory budget: retried by a launch with the full-size layout
            if (lane == 0) B.overflow_list[atomicAdd(B.n_overflow, 1)] = sample;
            continue;
        }
        if (!certified) {
            if (!B.final_pass) {
                if (lane == 0) {
                    B.status[sample] = kStatusNeedsMoreAdmm;
                    const int slot = atomicAdd(B.n_failed, 1);
                    B.failed_list[slot] = sample;
                }
                continue;
            }
            if (B.final_pass == 2) {
                // after the float64 fallback: no certificate, no answer (undecided, never an unproven "solved")
                if (lane == 0) {
                    B.status[sample] = CARMPC_QP_MAX_ITER;
                    if (B.u0) { B.u0[sample] = NaN; B.u0[B.stride + sample] = NaN; }
                    if (B.objective) B.objective[sample] = NaN;
                    if (B.polished) B.polished[sample] = 0;
                    if (B.stats) atomicAdd(B.stats + 19, 1ull);
                }
                if (B.u_full) for (int j = lane; j < n; j += 32) B.u_full[(size_t)sample * n + j] = NaN;
                continue;
            }
            if (B.stats && lane == 0 && B.rounds != 0) atomicAdd(B.stats + 16, 1ull);
            // the float32 ADMM iterate, objective 1/2 u'Hu + q'u evaluated directly: what opts.polish = 0 returns, and a
            // placeholder (polished = 0) for samples that the float64 fallback (qp_exact.cu) settles next
            for (int j = lane; j < n; j += 32) u[j] = (double)B.u_admm[(size_t)sample * n + j];
            __syncwarp();
            double part = 0.0;
            for (int j = lane; j < n; j += 32) {
                const double* f = T.F + (size_t)j * 4;
                const double qj = f[0] * dx[0] + f[1] * dx[1] + f[2] * dx[2] + f[3] * dx[3];
                double s = 0;                                     // H is symmetric: column walk is coalesced
                for (int k = 0; k < n; ++k) s += T.H[(size_t)k * n + j] * u[k];
                part += u[j] * (0.5 * s + qj);
            }
            obj = warp_sum(part);
        } else {
            // at a KKT point  H u + q + A_act' lambda = 0  and  A_act u = b_act  (rows with a skipped pivot have
            // lambda = 0), hence  1/2 u'Hu + q'u = 1/2 (q'u - lambda'b_act)
            double part = 0.0;
            for (int j = lane; j < n; j += 32) {
                const double* f = T.F + (size_t)j * 4;
                part += (f[0] * dx[0] + f[1] * dx[1] + f[2] * dx[2] + f[3] * dx[3]) * u[j];
            }
            for (int a = lane; a < na; a += 32) part -= rhs[a] * bact[a];
            obj = 0.5 * warp_sum(part);
        }
        if (lane == 0) {
            if (B.u0) { B.u0[sample] = u[0]; B.u0[B.stride + sample] = n > 1 ? u[1] : 0.0; }
            if (B.objective) B.objective[sample] = obj;
            if (B.polished) B.polished[sample] = certified ? 1 : 0;
            if (certified) B.status[sample] = CARMPC_QP_SOLVED;
            if (certified && B.iters_out) B.iters_out[sample] = 0;
            if (certified && B.final_pass == 2 && B.stats) atomicAdd(B.stats + 17, 1ull);
        }
        if (certified && B.sign_out) for (int i = lane; i < mt; i += 32) B.sign_out[(size_t)sample * mt + i] = sgn[i];
        if (B.u_full) for (int j = lane; j < n; j += 32) B.u_full[(size_t)sample * n + j] = u[j];
        // the multipliers this certificate checked (the row was zeroed by the entry point: only active rows are written)
        if (certified && B.cert) {
            double* row = B.cert + (size_t)sample * (mt + T.kpre);
            for (int a = lane; a < na; a += 32) { const int i = act[a]; row[i] = i < m ? T.rsign[i] * rhs[a] : rhs[a]; }
        }
        // Anchor of a seeded map: export the active rows and the affine multiplier map lambda(x0) = Lam [x0; 1] of this
        // critical region (five more right-hand sides through the factor already in shared memory).
        if (certified && b_rec_write && B.cdist == nullptr) {
            const int rec = B.rec_of[sample];
            if (rec >= 0 && na <= kPolishSmallActive) {
                for (int c = 0; c < 5; ++c) {
                    __syncwarp();
                    for (int a = lane; a < na; a += 32) {
                        const int i = act[a];
                        const double* w = T.AUu + (size_t)i * 4;
                        double v;
                        if (c < 4) v = w[c] + (i < m ? T.Gx[(size_t)i * 4 + c] : 0.0);
                        else v = -(w[0] * B.xref[0] + w[1] * B.xref[1] + w[2] * B.xref[2] + w[3] * B.xref[3]) - (sgn[i] > 0 ? T.hi[i] : T.lo[i]);
                        rhs[a] = v;
                    }
                    __syncwarp();
                    solve_in_place();
                    for (int a = lane; a < na; a += 32) B.rec_lam[((size_t)rec * kPolishSmallActive + a) * 5 + c] = rhs[a];
                }
                for (int a = lane; a < na; a += 32) B.rec_act[(size_t)rec * (kPolishSmallActive + 1) + 1 + a] = act[a];
                if (lane == 0) B.rec_act[(size_t)rec * (kPolishSmallActive + 1)] = na;
            }
        }
    }
}

// Exact Farkas certificates from the ADMM state.  The ADMM dual iterate of an infeasible problem grows along a Farkas
// direction; taken as it is (y = E (w - clip(w)) from the stored ADMM state, box multipliers y_b = -G'y so that A'y = 0 holds
// exactly) it is a certificate whenever its support value is negative - and that value is affine in the state.
//   mode 0 (anchors of a seeded map, status infeasible): store cx[4], c0, |cx|-bound[4], |c0|-bound in the anchor's
//          multiplier-map slot (type tag -2); a follower evaluates S(x0) = c0 - cx.x0 < -1e-9 (A0 + Ax.|x0|).
//   mode 1 (samples that ran out of ADMM iterations): a valid certificate turns "max_iter" into a proven "infeasible".
//   mode 2 (samples the first pass could not settle: iteration cap hit, or active set not certified): the same test
//          before the second pass; proven-infeasible samples are done, the others are listed for the tighter ADMM pass
//          (barely infeasible states are most of that list, and they are the ones that iterate longest).
// One warp per sample.
struct FarkasArgs {
    const int* list; int count; const int* count_dev; int mode;
    int* status; const float* warm; const double* x0; int64_t stride;
    const double* cdist;                                               // nullable per-sample disturbance
    const int* rec_of; double* rec_lam; int* rec_act;                  // mode 0
    double* cert;                                                      // nullable: rows of proven samples (mode 0: anchors)
    double* u0; double* objective; double* u_full; int8_t* polished;   // mode 1, 2 (nullable)
    int* survivors; int* n_survivors;                                  // mode 2
    unsigned long long* stats;
};

// CERT: the certificate store is a separate instantiation, so that a solve without certificates runs the same code as before
template <bool CERT>
__global__ void __launch_bounds__(128) farkas_kernel(const PolishTables T, const FarkasArgs F) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int n = T.n, m = T.m, mt = T.mt;
    double* y = reinterpret_cast<double*>(smem_raw) + (size_t)warp * m;
    const int gw = blockIdx.x * 4 + warp, nw = gridDim.x * 4;
    const int f_count = F.count_dev != nullptr ? min(*F.count_dev, F.count) : F.count;
    for (int q = gw; q < f_count; q += nw) {
        const int sample = F.list ? F.list[q] : q;
        const int rec = F.mode == 0 ? F.rec_of[sample] : 0;
        const int want = F.mode == 0 ? CARMPC_QP_INFEASIBLE : (F.mode == 1 ? CARMPC_QP_MAX_ITER : kStatusNeedsMoreAdmm);
        if (F.status[sample] != want || rec < 0) continue;
        double x0[4];
#pragma unroll
        for (int c = 0; c < 4; ++c) x0[c] = F.x0[(size_t)c * F.stride + sample];
        const double cd = F.cdist ? F.cdist[sample] : 0.0;

        double c0 = 0.0, A0 = 0.0, cx[4] = {0, 0, 0, 0}, Ax[4] = {0, 0, 0, 0};
        __syncwarp();
        for (int i = lane; i < m; i += 32) {
            const double* gx = T.Gx + (size_t)i * 4;
            const double dshift = T.Gc[i] * cd;                        // the per-sample disturbance moves the bounds
            const double shift = gx[0] * x0[0] + gx[1] * x0[1] + gx[2] * x0[2] + gx[3] * x0[3] + dshift;
            const double e = T.Eg[i], hi = T.hi[i], lo = T.lo[i];
            const double w = (double)F.warm[(size_t)sample * mt + i];
            const double hs = e * (hi - shift), ls = e * (lo - shift);
            double yu = 0.0;
            if (isfinite(w)) yu = e * (w > hs ? w - hs : (w < ls ? w - ls : 0.0));
            y[i] = yu;
            if (yu != 0.0) {
                const double t = ((yu > 0.0 ? hi : lo) - dshift) * yu;
                c0 += t; A0 += fabs(t) + fabs(dshift * yu);
#pragma unroll
                for (int c = 0; c < 4; ++c) { cx[c] += yu * gx[c]; Ax[c] += fabs(yu * gx[c]); }
            }
        }
        __syncwarp();
        for (int j = lane; j < n; j += 32) {
            double s = 0.0;
            for (int i = 0; i < m; ++i) s += T.G[(size_t)i * n + j] * y[i];
            const double yb = -s;
            if (yb != 0.0) {
                const double t = (yb > 0.0 ? T.hi[m + j] : T.lo[m + j]) * yb;
                c0 += t; A0 += fabs(t);
            }
        }
        c0 = warp_sum(c0); A0 = warp_sum(A0);
#pragma unroll
        for (int c = 0; c < 4; ++c) { cx[c] = warp_sum(cx[c]); Ax[c] = warp_sum(Ax[c]); }
        const double S = c0 - (cx[0] * x0[0] + cx[1] * x0[1] + cx[2] * x0[2] + cx[3] * x0[3]);
        const double margin = 1e-9 * (A0 + Ax[0] * fabs(x0[0]) + Ax[1] * fabs(x0[1]) + Ax[2] * fabs(x0[2]) + Ax[3] * fabs(x0[3]));
        const bool valid = isfinite(S) && isfinite(margin) && S < -margin;
        if (!valid) {
            if (F.mode == 2 && lane == 0) F.survivors[atomicAdd(F.n_survivors, 1)] = sample;
            continue;
        }
        if (CERT) {
            // y as tested above, box part recomputed by the same expression (a mode-0 row replaces the anchor's own proof:
            // it is the certificate its followers' support values S(x0) use)
            double* row = F.cert + (size_t)sample * (mt + T.kpre);
            for (int i = lane; i < m; i += 32) row[i] = T.rsign[i] * y[i];
            for (int j = lane; j < n; j += 32) {
                double s = 0.0;
                for (int i = 0; i < m; ++i) s += T.G[(size_t)i * n + j] * y[i];
                row[m + j] = -s;
            }
            for (int k = lane; k < T.kpre; k += 32) row[mt + k] = 0.0;
        }
        if (F.mode == 0) {
            if (lane == 0) {
                double* r = F.rec_lam + (size_t)rec * kPolishSmallActive * 5;
                r[0] = cx[0]; r[1] = cx[1]; r[2] = cx[2]; r[3] = cx[3]; r[4] = c0;
                r[5] = Ax[0]; r[6] = Ax[1]; r[7] = Ax[2]; r[8] = Ax[3]; r[9] = A0;
                F.rec_act[(size_t)rec * (kPolishSmallActive + 1)] = -2;
            }
        } else {
            const double NaN = __longlong_as_double(0x7ff8000000000000ll);
            if (lane == 0) {
                F.status[sample] = CARMPC_QP_INFEASIBLE;
                if (F.u0) { F.u0[sample] = NaN; F.u0[F.stride + sample] = NaN; }
                if (F.objective) F.objective[sample] = INFINITY;
                if (F.polished) F.polished[sample] = 0;
                if (F.stats) atomicAdd(F.stats + (F.mode == 1 ? 14 : 15), 1ull);
            }
            if (F.u_full) for (int j = lane; j < n; j += 32) F.u_full[(size_t)sample * n + j] = NaN;
        }
    }
}

}  // namespace

static int farkas_launch(QPHandle* qh, const FarkasArgs& f, cudaStream_t st) {
    if (f.count <= 0) return CARMPC_OK;
    const size_t smem = sizeof(double) * 4 * (size_t)qh->polish.m;
    const int blocks = (int)std::max<int64_t>(1, std::min<int64_t>((f.count + 3) / 4, (int64_t)qh->sm * 8));
    if (f.cert) farkas_kernel<true><<<blocks, 128, smem, st>>>(qh->polish, f);
    else farkas_kernel<false><<<blocks, 128, smem, st>>>(qh->polish, f);
    CARMPC_CUDA(cudaGetLastError());
    return CARMPC_OK;
}

// the per-sample arrays, the histogram and the certificate rows of the call
static FarkasArgs farkas_args(const PolishBatch& b, const int* d_list, int count, const int* d_count, int mode,
                              const float* d_warm) {
    FarkasArgs f = {};
    f.list = d_list; f.count = count; f.count_dev = d_count; f.mode = mode; f.status = b.status; f.warm = d_warm;
    f.x0 = b.x0; f.stride = b.stride; f.cdist = b.cdist;
    f.u0 = b.u0; f.objective = b.objective; f.u_full = b.u_full; f.polished = b.polished; f.stats = b.stats; f.cert = b.cert;
    return f;
}

int farkas_export_launch(QPHandle* qh, const PolishBatch& b, const int* d_list, int count, const float* d_warm, cudaStream_t st) {
    FarkasArgs f = farkas_args(b, d_list, count, nullptr, 0, d_warm);
    f.rec_of = b.rec_of; f.rec_lam = b.rec_lam; f.rec_act = b.rec_act;
    return farkas_launch(qh, f, st);
}

int farkas_decide_launch(QPHandle* qh, const PolishBatch& b, const int* d_list, int count, const int* d_count,
                         const float* d_warm, cudaStream_t st) {
    return farkas_launch(qh, farkas_args(b, d_list, count, d_count, 1, d_warm), st);
}

int farkas_filter_launch(QPHandle* qh, const PolishBatch& b, const int* d_list, int count, const float* d_warm,
                         int* d_survivors, int* d_n_survivors, cudaStream_t st) {
    FarkasArgs f = farkas_args(b, d_list, count, nullptr, 2, d_warm);
    f.survivors = d_survivors; f.n_survivors = d_n_survivors;
    return farkas_launch(qh, f, st);
}

// ---- the empty active set, tried first ----------------------------------------------------------------------------------
// If the unconstrained minimiser u = -H^-1 F (x0 - xref) = Uu dx satisfies every row (same float64 expressions and the same
// tolerance as the KKT certificate above with no active row), it IS the optimum: one thread per sample, ~9 DFMA per row, no
// factorisation, no iteration.  That is the common case of a closed loop once the run is near its goal (LQR region), and a
// few per cent of a region-of-attraction grid.  Samples it cannot settle are listed for the regular pipeline.
struct UnconstrainedArgs {
    const double* x0; int64_t stride; const double* cdist; double xref[4];
    const int* list; int count; const int* count_dev;
    int* status; double* u0; double* objective; double* u_full; int8_t* polished; int8_t* sign; int* iters_out;
    unsigned long long* stats;
    int* rest_list; int* n_rest;
    const double* Px; const double* Pc; const double* pre_lo; const double* pre_hi; int kpre;
};

__global__ void __launch_bounds__(256) polish_unconstrained_kernel(const PolishTables T, const UnconstrainedArgs A) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int n = T.n, m = T.m, mt = T.mt;
    double* s_auu = reinterpret_cast<double*>(smem_raw);      // [mt][4]
    double* s_gx = s_auu + (size_t)mt * 4;                    // [m][4]
    double* s_gc = s_gx + (size_t)m * 4;                      // [m]
    double* s_hi = s_gc + m;                                  // [mt]
    double* s_lo = s_hi + mt;                                 // [mt]
    for (int i = threadIdx.x; i < mt * 4; i += blockDim.x) s_auu[i] = T.AUu[i];
    for (int i = threadIdx.x; i < m * 4; i += blockDim.x) s_gx[i] = T.Gx[i];
    for (int i = threadIdx.x; i < m; i += blockDim.x) s_gc[i] = T.Gc[i];
    for (int i = threadIdx.x; i < mt; i += blockDim.x) { s_hi[i] = T.hi[i]; s_lo[i] = T.lo[i]; }
    __syncthreads();
    const int count = A.count_dev ? min(*A.count_dev, A.count) : A.count;
    const int lane = threadIdx.x & 31;
    const int rounds = (count + gridDim.x * blockDim.x - 1) / (gridDim.x * blockDim.x);
    for (int r = 0; r < rounds; ++r) {
        const int q = (r * gridDim.x + blockIdx.x) * blockDim.x + threadIdx.x;
        const bool have = q < count;
        int sample = 0;
        bool ok = false;
        double dx[4] = {0.0, 0.0, 0.0, 0.0};
        if (have) {
            sample = A.list ? A.list[q] : q;
            double x0[4];
#pragma unroll
            for (int c = 0; c < 4; ++c) { x0[c] = A.x0[(size_t)c * A.stride + sample]; dx[c] = x0[c] - A.xref[c]; }
            const double cd = A.cdist ? A.cdist[sample] : 0.0;
            ok = isfinite(x0[0]) && isfinite(x0[1]) && isfinite(x0[2]) && isfinite(x0[3]);
            for (int k = 0; k < A.kpre; ++k) {
                const double v = A.Px[k * 4 + 0] * x0[0] + A.Px[k * 4 + 1] * x0[1] + A.Px[k * 4 + 2] * x0[2] +
                                 A.Px[k * 4 + 3] * x0[3] + A.Pc[k] * cd;
                ok = ok && v <= A.pre_hi[k] && v >= A.pre_lo[k];
            }
            double worst = 0.0;
            if (ok) {
                for (int i = 0; i < mt; ++i) {
                    const double* w = s_auu + i * 4;
                    double t = w[0] * dx[0] + w[1] * dx[1] + w[2] * dx[2] + w[3] * dx[3];
                    if (i < m) {
                        const double* gx = s_gx + i * 4;
                        t += gx[0] * x0[0] + gx[1] * x0[1] + gx[2] * x0[2] + gx[3] * x0[3] + s_gc[i] * cd;
                    }
                    const double h = s_hi[i], l = s_lo[i];
                    if (isinf(h) && isinf(l)) continue;
                    worst = fmax(worst, fmax(t - h, l - t));
                }
                ok = worst <= kFeasTol;                       // NaN compares false
            }
            if (ok) {
                const double u0 = T.Uu[0] * dx[0] + T.Uu[1] * dx[1] + T.Uu[2] * dx[2] + T.Uu[3] * dx[3];
                const double u1 = n > 1 ? T.Uu[4] * dx[0] + T.Uu[5] * dx[1] + T.Uu[6] * dx[2] + T.Uu[7] * dx[3] : 0.0;
                if (A.u0) { A.u0[sample] = u0; A.u0[A.stride + sample] = u1; }
                if (A.objective || A.u_full) {
                    double part = 0.0;                        // 1/2 q'u at the unconstrained optimum (H u + q = 0)
                    for (int j = 0; j < n; ++j) {
                        const double* w = T.Uu + (size_t)j * 4;
                        const double* f = T.F + (size_t)j * 4;
                        const double uj = w[0] * dx[0] + w[1] * dx[1] + w[2] * dx[2] + w[3] * dx[3];
                        part += (f[0] * dx[0] + f[1] * dx[1] + f[2] * dx[2] + f[3] * dx[3]) * uj;
                        if (A.u_full) A.u_full[(size_t)sample * n + j] = uj;
                    }
                    if (A.objective) A.objective[sample] = 0.5 * part;
                }
                A.status[sample] = CARMPC_QP_SOLVED;
                if (A.polished) A.polished[sample] = 1;
                if (A.iters_out) A.iters_out[sample] = 0;
            } else {
                A.rest_list[atomicAdd(A.n_rest, 1)] = sample;
            }
        }
        // the certified (empty) active set replaces whatever the workspace held for the sample: one row per lane in turn,
        // zeroed by the whole warp (coalesced byte stores)
        const unsigned done = __ballot_sync(0xffffffffu, have && ok);
        if (A.sign != nullptr) {
            unsigned todo = done;
            while (todo) {
                const int src = __ffs(todo) - 1;
                todo &= todo - 1;
                const int s2 = __shfl_sync(0xffffffffu, sample, src);
                for (int i = lane; i < mt; i += 32) A.sign[(size_t)s2 * mt + i] = 0;
            }
        }
        if (A.stats && lane == 0 && done) atomicAdd(A.stats + 0, (unsigned long long)__popc(done));
    }
}

// d_rest / d_n_rest (zeroed here) receive the samples the empty set does not settle
int polish_unconstrained_launch(QPHandle* qh, const PolishBatch& b, int* d_rest, int* d_n_rest, cudaStream_t st) {
    if (b.count <= 0) return CARMPC_OK;
    UnconstrainedArgs a;
    memset(&a, 0, sizeof(a));
    a.x0 = b.x0; a.stride = b.stride; a.cdist = b.cdist;
    for (int c = 0; c < 4; ++c) a.xref[c] = b.xref[c];
    a.list = b.idx_list; a.count = b.count; a.count_dev = b.count_dev;
    a.status = b.status; a.u0 = b.u0; a.objective = b.objective; a.u_full = b.u_full; a.polished = b.polished;
    a.sign = b.sign_out; a.iters_out = b.iters_out; a.stats = b.stats;
    a.rest_list = d_rest; a.n_rest = d_n_rest;
    a.Px = qh->admm.Px; a.Pc = qh->admm.Pc; a.pre_lo = qh->admm.pre_lo; a.pre_hi = qh->admm.pre_hi; a.kpre = qh->admm.kpre;
    CARMPC_CUDA(cudaMemsetAsync(d_n_rest, 0, sizeof(int), st));
    const int n = qh->polish.n, m = qh->polish.m, mt = qh->polish.mt;
    (void)n;
    const size_t smem = sizeof(double) * ((size_t)mt * 4 + (size_t)m * 5 + (size_t)mt * 2);
    { const int rc = kernel_config(reinterpret_cast<const void*>(polish_unconstrained_kernel), 256, smem, nullptr); if (rc != CARMPC_OK) return rc; }
    const int blocks = (int)std::max<int64_t>(1, std::min<int64_t>(((int64_t)b.count + 255) / 256, (int64_t)qh->sm * 4));
    polish_unconstrained_kernel<<<blocks, 256, smem, st>>>(qh->polish, a);
    CARMPC_CUDA(cudaGetLastError());
    return CARMPC_OK;
}

static int polish_launch_cap(QPHandle* qh, const PolishBatch& b, cudaStream_t st) {
    const PolishSmemLayout L = polish_layout(qh->polish.n, qh->polish.mt, b.na_cap);
    constexpr int warps = kPolishThreads / 32;
    const size_t smem = L.per_warp * warps;
    if (smem > (size_t)227 * 1024) { set_error("polish: shared-memory budget exceeded"); return CARMPC_ERR_UNSUPPORTED; }
    void (*kernel)(const PolishTables, const PolishBatch);
    if (b.seed != nullptr) kernel = polish_kernel<true, true, false>;
    else if (b.precheck) kernel = polish_kernel<false, true, false>;
    else if (b.rec_write) kernel = polish_kernel<false, false, true>;
    else kernel = polish_kernel<false, false, false>;
    int per_sm = 0;
    { const int rc = kernel_config(reinterpret_cast<const void*>(kernel), kPolishThreads, smem, &per_sm); if (rc != CARMPC_OK) return rc; }
    const int64_t need = (b.count + warps - 1) / warps;
    const int blocks = (int)std::max<int64_t>(1, std::min<int64_t>(need, (int64_t)qh->sm * per_sm));
    kernel<<<blocks, kPolishThreads, smem, st>>>(qh->polish, b);
    CARMPC_CUDA(cudaGetLastError());
    return CARMPC_OK;
}

// Two launches: a small active-set budget (32 rows: 7 KB of shared memory per warp, 28 warps per SM) covers almost
// every sample; the few with more active rows are listed and redone with the full-size layout.
int polish_launch(QPHandle* qh, const PolishBatch& b_in, cudaStream_t st) {
    if (b_in.count <= 0) return CARMPC_OK;
    const int n = qh->polish.n, mt = qh->polish.mt;
    const int full = std::min(mt, std::min(kPolishMaxActive, n + 8));
    PolishBatch b = b_in;
    if (full <= kPolishSmallActive || qh->ws_overflow == nullptr) {
        b.na_cap = full; b.overflow_list = nullptr; b.n_overflow = nullptr;
        return polish_launch_cap(qh, b, st);
    }
    CARMPC_CUDA(cudaMemsetAsync(qh->ws_counters + kCntOverflow, 0, sizeof(int), st));
    b.na_cap = kPolishSmallActive; b.overflow_list = qh->ws_overflow; b.n_overflow = qh->ws_counters + kCntOverflow;
    int rc = polish_launch_cap(qh, b, st);
    if (rc != CARMPC_OK) return rc;
    // the overflow launch reads its sample count on the device (no host round trip; with nothing listed its CTAs exit at once)
    b.na_cap = full; b.idx_list = qh->ws_overflow; b.count_dev = qh->ws_counters + kCntOverflow; b.overflow_list = nullptr; b.n_overflow = nullptr;
    return polish_launch_cap(qh, b, st);
}

}  // namespace carmpc
