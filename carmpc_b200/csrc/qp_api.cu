// C ABI of the batched QP solver (include/carmpc.h, part B): handle creation (host setup + upload), the two-pass
// ADMM -> polish orchestration, host-buffer convenience entry point and statistics.
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>

#include "qp_internal.cuh"

namespace carmpc {

namespace {

template <class T>
int upload(QPHandle* q, const std::vector<T>& v, const T** dst) {
    void* d = nullptr;
    const size_t bytes = sizeof(T) * std::max<size_t>(v.size(), 1);
    CARMPC_CUDA(cudaMalloc(&d, bytes));
    q->allocations.push_back(d);
    if (!v.empty()) CARMPC_CUDA(cudaMemcpy(d, v.data(), sizeof(T) * v.size(), cudaMemcpyHostToDevice));
    *dst = static_cast<const T*>(d);
    return CARMPC_OK;
}

__global__ void aos_to_soa_kernel(const double* __restrict__ aos, double* __restrict__ soa, int64_t count, int width) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    for (int c = 0; c < width; ++c) soa[(size_t)c * count + i] = aos[i * width + c];
}

__global__ void soa_to_aos_kernel(const double* __restrict__ soa, double* __restrict__ aos, int64_t count, int width) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    for (int c = 0; c < width; ++c) aos[i * width + c] = soa[(size_t)c * count + i];
}

// seeded solve: anchors are the samples that name themselves (or nothing valid) as their seed; a follower's seed must be
// an anchor (single level), anything else is solved cold as well
__global__ void split_seeds_kernel(const int* __restrict__ seed, int count, int* __restrict__ anchors, int* __restrict__ followers,
                                   int* __restrict__ counters, int* __restrict__ rec_of) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    bool follow = false;
    if (i < count) {
        const int s = seed[i];
        if (s >= 0 && s < count && s != i) { const int ss = seed[s]; follow = ss == s || ss < 0 || ss >= count; }
    }
    // order-preserving within a warp; warps append in arrival order (the lists only drive work queues)
    const unsigned fm = __ballot_sync(0xffffffffu, i < count && follow), am = __ballot_sync(0xffffffffu, i < count && !follow);
    const int lane = threadIdx.x & 31;
    int fb = 0, abase = 0;
    if (lane == 0) { if (fm) fb = atomicAdd(counters + 1, __popc(fm)); if (am) abase = atomicAdd(counters + 0, __popc(am)); }
    fb = __shfl_sync(0xffffffffu, fb, 0); abase = __shfl_sync(0xffffffffu, abase, 0);
    if (i < count) {
        const unsigned below = (1u << lane) - 1u;
        if (follow) {
            followers[fb + __popc(fm & below)] = i;
            rec_of[i] = -1;
        } else {
            const int pos = abase + __popc(am & below);
            anchors[pos] = i;
            rec_of[i] = pos;                 // an anchor's record (multiplier map of its critical region) sits at its list position
        }
    }
}

// region-of-attraction map: expand the C-order tensor grid into SoA states and name every point's lattice anchor (the
// centre of its block of `block` points per axis)
struct MapGrid {
    int dims[4], state_of_axis[4], offset[4], block[4];
};

__global__ void map_expand_kernel(const double* __restrict__ axes, MapGrid g, int64_t n, double* __restrict__ x0, int* __restrict__ seed) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    int64_t rem = i, anchor = 0, stride = n;
    for (int k = 0; k < 4; ++k) {
        stride /= g.dims[k];
        const int idx = (int)(rem / stride);
        rem -= (int64_t)idx * stride;
        x0[(size_t)g.state_of_axis[k] * n + i] = axes[g.offset[k] + idx];
        const int b = g.block[k];
        const int centre = min((idx / b) * b + b / 2, g.dims[k] - 1);
        anchor += (int64_t)centre * stride;
    }
    seed[i] = (int)anchor;
}

// The base values of a request's polish and ADMM launches (both pipelines): every stage then sets its own list, counters and
// pass-specific fields on a copy.
PolishBatch polish_batch(QPHandle& q, const SolveRequest& r) {
    PolishBatch pb;
    memset(&pb, 0, sizeof(pb));
    pb.x0 = r.x0; pb.stride = r.stride; pb.cdist = r.c;
    for (int c = 0; c < 4; ++c) pb.xref[c] = r.xref[c];
    pb.idx_list = r.idx; pb.count = (int)r.count; pb.count_dev = r.count_dev;
    pb.sign = q.ws_sign; pb.u_admm = q.ws_u; pb.status = r.status ? r.status : q.ws_status;
    pb.u0 = r.u0; pb.objective = r.objective; pb.u_full = r.u_full; pb.polished = q.ws_polished;
    pb.n_failed = q.ws_counters + kCntFailed; pb.failed_list = q.ws_failed;
    pb.rounds = q.host.opts.polish ? -1 : 0; pb.final_pass = q.host.opts.polish ? 0 : 1;
    pb.stats = q.ws_polish_stats; pb.cert = r.cert;
    // warm-started sequences and seeded maps keep the certified (repaired) active set
    if ((r.warm && r.warm_out) || r.keep_sign) pb.sign_out = q.ws_sign;
    if (r.records) {
        pb.rec_of = q.ws_rec_of; pb.rec_lam = q.ws_rec_lam; pb.rec_act = q.ws_rec_act;
        pb.rec_write = r.seed == nullptr;                 // anchors export, followers read (p0 in solve)
    }
    return pb;
}

AdmmBatch admm_batch(QPHandle& q, const SolveRequest& r) {
    AdmmBatch ab;
    memset(&ab, 0, sizeof(ab));
    ab.x0 = r.x0; ab.stride = r.stride; ab.cdist = r.c;
    for (int c = 0; c < 4; ++c) ab.xref[c] = r.xref[c];
    ab.idx_list = r.idx; ab.count = (int)r.count; ab.count_dev = r.count_dev; ab.next = q.ws_counters + kCntNext;
    ab.sign = q.ws_sign; ab.u_admm = q.ws_u; ab.status = r.status ? r.status : q.ws_status; ab.iters = r.iters ? r.iters : q.ws_iters;
    // the ADMM state of every sample is kept (caller's buffer or the workspace): the second pass resumes from it
    ab.warm = r.warm ? r.warm : q.ws_warm; ab.warm_in = r.warm ? r.warm_in : 0; ab.warm_out = 1;
    ab.total_iters = q.ws_total_iters; ab.eps_scale = 1.f; ab.max_iter = q.host.opts.max_iter;
    return ab;
}

// Results of the host-buffer entry points: u0 back to the caller's (batch x 2) layout, the rest as it is; synchronises.
int download(QPHandle* q, int64_t batch, double* h_u0, double* h_objective, int32_t* h_status, int32_t* h_iters,
             double* h_u_full, cudaStream_t st) {
    if (h_u0) {
        soa_to_aos_kernel<<<(int)((batch + 255) / 256), 256, 0, st>>>(q->io_u0, q->io_u0_aos, batch, 2);
        CARMPC_CUDA(cudaMemcpyAsync(h_u0, q->io_u0_aos, sizeof(double) * 2 * batch, cudaMemcpyDeviceToHost, st));
    }
    if (h_objective) CARMPC_CUDA(cudaMemcpyAsync(h_objective, q->io_obj, sizeof(double) * batch, cudaMemcpyDeviceToHost, st));
    CARMPC_CUDA(cudaMemcpyAsync(h_status, q->io_status, sizeof(int32_t) * batch, cudaMemcpyDeviceToHost, st));
    if (h_iters) CARMPC_CUDA(cudaMemcpyAsync(h_iters, q->io_iters, sizeof(int32_t) * batch, cudaMemcpyDeviceToHost, st));
    if (h_u_full) CARMPC_CUDA(cudaMemcpyAsync(h_u_full, q->io_full, sizeof(double) * (size_t)q->host.n * batch, cudaMemcpyDeviceToHost, st));
    CARMPC_CUDA(cudaStreamSynchronize(st));
    CARMPC_CUDA(cudaGetLastError());
    return CARMPC_OK;
}

}  // namespace

int QPHandle::ensure_io(int64_t batch, bool want_full) {
    if (batch > io_cap) {
        cudaFree(io_x0_aos); cudaFree(io_x0); cudaFree(io_c); cudaFree(io_u0); cudaFree(io_u0_aos); cudaFree(io_obj);
        cudaFree(io_status); cudaFree(io_iters); cudaFree(io_seed);
        io_seed = nullptr;
        io_x0_aos = io_x0 = io_c = io_u0 = io_u0_aos = io_obj = nullptr; io_status = io_iters = nullptr;
        io_cap = 0;
        CARMPC_CUDA(cudaMalloc(&io_x0_aos, sizeof(double) * 4 * batch));
        CARMPC_CUDA(cudaMalloc(&io_x0, sizeof(double) * 4 * batch));
        CARMPC_CUDA(cudaMalloc(&io_c, sizeof(double) * batch));
        CARMPC_CUDA(cudaMalloc(&io_u0, sizeof(double) * 2 * batch));
        CARMPC_CUDA(cudaMalloc(&io_u0_aos, sizeof(double) * 2 * batch));
        CARMPC_CUDA(cudaMalloc(&io_obj, sizeof(double) * batch));
        CARMPC_CUDA(cudaMalloc(&io_status, sizeof(int32_t) * batch));
        CARMPC_CUDA(cudaMalloc(&io_iters, sizeof(int32_t) * batch));
        CARMPC_CUDA(cudaMalloc(&io_seed, sizeof(int32_t) * batch));
        io_cap = batch;
    }
    if (want_full && batch > io_full_cap) {
        cudaFree(io_full); io_full = nullptr; io_full_cap = 0;
        CARMPC_CUDA(cudaMalloc(&io_full, sizeof(double) * (size_t)host.n * batch));
        io_full_cap = batch;
    }
    return CARMPC_OK;
}

QPHandle::~QPHandle() {
    for (void* p : allocations) cudaFree(p);
    cudaFree(ws_sign); cudaFree(ws_u); cudaFree(ws_status); cudaFree(ws_iters); cudaFree(ws_failed); cudaFree(ws_failed0); cudaFree(ws_rest);
    cudaFree(ws_counters); cudaFree(ws_total_iters); cudaFree(ws_polished); cudaFree(ws_warm); cudaFree(ws_overflow); cudaFree(ws_unproven);
    cudaFree(ws_anchor); cudaFree(ws_follow); cudaFree(ws_rec_of); cudaFree(ws_rec_lam); cudaFree(ws_rec_act); cudaFree(ws_polish_stats);
    cudaFree(io_x0_aos); cudaFree(io_x0); cudaFree(io_c); cudaFree(io_u0); cudaFree(io_u0_aos); cudaFree(io_obj); cudaFree(io_full);
    cudaFree(io_status); cudaFree(io_iters); cudaFree(io_seed); cudaFree(io_axes); cudaFree(ws_prof);
}

int QPHandle::ensure_workspace(int64_t batch) {
    if (ws_counters == nullptr) {
        CARMPC_CUDA(cudaMalloc(&ws_counters, sizeof(int) * kCounters));
        CARMPC_CUDA(cudaMalloc(&ws_total_iters, sizeof(unsigned long long)));
        CARMPC_CUDA(cudaMalloc(&ws_polish_stats, sizeof(unsigned long long) * kPolishStats));
        CARMPC_CUDA(cudaMemset(ws_polish_stats, 0, sizeof(unsigned long long) * kPolishStats));
    }
    if (batch <= ws_batch) return CARMPC_OK;
    cudaFree(ws_sign); cudaFree(ws_u); cudaFree(ws_status); cudaFree(ws_iters); cudaFree(ws_failed); cudaFree(ws_polished);
    cudaFree(ws_warm); ws_warm = nullptr;
    cudaFree(ws_overflow); ws_overflow = nullptr;
    cudaFree(ws_unproven); ws_unproven = nullptr;
    cudaFree(ws_failed0); ws_failed0 = nullptr;
    cudaFree(ws_rest); ws_rest = nullptr;
    cudaFree(ws_anchor); ws_anchor = nullptr;
    cudaFree(ws_follow); ws_follow = nullptr;
    cudaFree(ws_rec_of); ws_rec_of = nullptr;
    ws_sign = nullptr; ws_u = nullptr; ws_status = nullptr; ws_iters = nullptr; ws_failed = nullptr; ws_polished = nullptr;
    ws_batch = 0;
    CARMPC_CUDA(cudaMalloc(&ws_sign, (size_t)batch * admm.mt));
    CARMPC_CUDA(cudaMalloc(&ws_u, sizeof(float) * (size_t)batch * admm.n));
    CARMPC_CUDA(cudaMalloc(&ws_status, sizeof(int) * (size_t)batch));
    CARMPC_CUDA(cudaMalloc(&ws_iters, sizeof(int) * (size_t)batch));
    CARMPC_CUDA(cudaMalloc(&ws_failed, sizeof(int) * (size_t)batch));
    CARMPC_CUDA(cudaMalloc(&ws_overflow, sizeof(int) * (size_t)batch));
    CARMPC_CUDA(cudaMalloc(&ws_unproven, sizeof(int) * (size_t)batch));
    CARMPC_CUDA(cudaMalloc(&ws_failed0, sizeof(int) * (size_t)batch));
    CARMPC_CUDA(cudaMalloc(&ws_rest, sizeof(int) * (size_t)batch));
    CARMPC_CUDA(cudaMalloc(&ws_anchor, sizeof(int) * (size_t)batch));
    CARMPC_CUDA(cudaMalloc(&ws_follow, sizeof(int) * (size_t)batch));
    CARMPC_CUDA(cudaMalloc(&ws_rec_of, sizeof(int) * (size_t)batch));
    CARMPC_CUDA(cudaMalloc(&ws_polished, (size_t)batch));
    CARMPC_CUDA(cudaMalloc(&ws_warm, sizeof(float) * (size_t)batch * admm.mt));
    ws_batch = batch;
    return CARMPC_OK;
}

int QPHandle::solve(const SolveRequest& r, cudaStream_t st, SolveCounts* counts) {
    if (host_only) { set_error("carmpc_qp: this handle was created without a CUDA device; there is no CPU solver"); return CARMPC_ERR_CUDA; }
    int rc = ensure_workspace(r.stride);
    if (rc != CARMPC_OK) return rc;
    SolveCounts own, &k = counts ? *counts : own;
    k = SolveCounts();
    last_tc_samples = 0;
    CARMPC_CUDA(cudaMemsetAsync(ws_counters, 0, sizeof(int) * 8, st));
    if (!r.keep_total) CARMPC_CUDA(cudaMemsetAsync(ws_total_iters, 0, sizeof(unsigned long long), st));
    PolishBatch pb = polish_batch(*this, r);
    AdmmBatch ab = admm_batch(*this, r);
    if (!r.hold_stats) CARMPC_CUDA(cudaMemsetAsync(ws_polish_stats, 0, sizeof(unsigned long long) * kPolishStats, st));

    // Active-set reuse (closed loop): consecutive QPs of a run mostly share their active set, so the set certified at
    // the previous step (kept in the workspace, same sample indexing) goes through the float64 polish first; only the
    // samples it does not certify (set changed, or infeasible now) run ADMM iterations.
    // The empty active set first (polish_unconstrained_kernel): where the unconstrained minimiser satisfies every row it is
    // the optimum - certified in float64 by one thread, no iteration, no factorisation.  Closed-loop runs near their goal
    // live there; on the config-3 grid it settles 8.6 % of the states.  The rest (listed on the device) goes on.
    if (host.opts.polish) {
        PolishBatch pu = pb;
        pu.sign_out = ws_sign; pu.iters_out = ab.iters;
        rc = polish_unconstrained_launch(this, pu, ws_rest, ws_counters + kCntRest, st);
        if (rc != CARMPC_OK) return rc;
        ++k.launches;
        pb.idx_list = ws_rest; pb.count_dev = ws_counters + kCntRest;
    }
    if (r.reuse && host.opts.polish) {
        PolishBatch p0 = pb;
        p0.rounds = 4; p0.final_pass = 0; p0.n_failed = ws_counters + kCntReuseFailed; p0.failed_list = ws_failed0;
        p0.precheck = 1; p0.Px = admm.Px; p0.Pc = admm.Pc; p0.pre_lo = admm.pre_lo; p0.pre_hi = admm.pre_hi; p0.kpre = admm.kpre;
        p0.sign_out = ws_sign; p0.iters_out = ab.iters; p0.seed = r.seed;
        p0.rec_write = 0; p0.rec_read = r.records && r.seed != nullptr;
        rc = polish_launch(this, p0, st);
        if (rc != CARMPC_OK) return rc;
        ++k.launches;
        int n_failed0 = 0;
        CARMPC_CUDA(cudaMemcpyAsync(&n_failed0, ws_counters + kCntReuseFailed, sizeof(int), cudaMemcpyDeviceToHost, st));
        CARMPC_CUDA(cudaStreamSynchronize(st));
        k.reused = r.count - n_failed0;
        if (n_failed0 == 0) { last_total_iters = 0; last_launches = k.launches; return CARMPC_OK; }   // no iteration
        pb.idx_list = ws_failed0; pb.count = n_failed0; pb.count_dev = nullptr;
    }

    ab.idx_list = pb.idx_list; ab.count = pb.count; ab.count_dev = pb.count_dev;
    // First pass capped at kFirstPassIters: on the region-of-attraction grid every solvable state converges within 90
    // iterations and only barely infeasible states run longer (up to ~400).  On 128-sample tiles such stragglers hold a
    // whole tile at ~10 us per iteration; handed to the second pass they continue on narrow tiles (~3 us per iteration).
    // The cap does not depend on the batch, so a state sees the same iteration schedule however it is batched (cold grid,
    // seeded map, alone): the statuses of cold solves are path-independent.  Warm-started solves (closed-loop steps: small
    // batches on narrow tiles, where a second pass only adds launches) keep the full budget.
    if (host.opts.polish && !(r.warm && r.warm_in))
        ab.max_iter = std::min(ab.max_iter, std::max(kFirstPassIters, admm.check_every));
    ab.write_u = host.opts.polish ? 0 : 1;        // with the polish on, only the final pass may fall back to the iterate
    rc = admm_launch(this, ab, st);
    if (rc != CARMPC_OK) return rc;
    ++k.launches;

    rc = polish_launch(this, pb, st);
    if (rc != CARMPC_OK) return rc;
    ++k.launches;

    int n_failed = 0;
    if (host.opts.polish) {
        // "infeasible" verdicts of the float32 ADMM are accepted only with a float64 Farkas certificate of their final
        // dual iterate (or a violated u-independent row); the others join the list of the second pass
        rc = farkas_verify_launch(this, pb, pb.idx_list, pb.count, pb.count_dev, ab.warm, ws_failed, ws_counters + kCntFailed, st);
        if (rc != CARMPC_OK) return rc;
        ++k.launches;
        CARMPC_CUDA(cudaMemcpyAsync(&n_failed, ws_counters + kCntFailed, sizeof(int), cudaMemcpyDeviceToHost, st));
        CARMPC_CUDA(cudaStreamSynchronize(st));
    }
    const int* second_list = ws_failed;
    // The certificate kernels take the disturbance shift as well; the public entry points keep their results with a
    // disturbance (max_iter instead of a certified "infeasible"), only the closed loop turns them on (certify_shifted).
    const bool certify = r.c == nullptr || r.certify_shifted;
    if (n_failed > 0 && certify) {
        // most of what the first pass could not settle is barely infeasible: the exact certificate test on the first-pass
        // state removes those before the (long) tighter pass
        CARMPC_CUDA(cudaMemsetAsync(ws_counters + kCntSurvivors, 0, sizeof(int), st));
        rc = farkas_filter_launch(this, pb, ws_failed, n_failed, ab.warm, ws_overflow, ws_counters + kCntSurvivors, st);
        if (rc != CARMPC_OK) return rc;
        ++k.launches;
        CARMPC_CUDA(cudaMemcpyAsync(&n_failed, ws_counters + kCntSurvivors, sizeof(int), cudaMemcpyDeviceToHost, st));
        CARMPC_CUDA(cudaStreamSynchronize(st));
        // the survivors move to ws_failed (the polish launches below reuse ws_overflow)
        if (n_failed > 0) CARMPC_CUDA(cudaMemcpyAsync(ws_failed, ws_overflow, sizeof(int) * n_failed, cudaMemcpyDeviceToDevice, st));
    }
    if (n_failed > 0) {
        // second pass on the samples whose active set the polish could not certify: tighter ADMM, then accept
        ab.idx_list = second_list; ab.count = n_failed; ab.count_dev = nullptr; ab.next = ws_counters + kCntNext2; ab.eps_scale = 0.01f;
        ab.max_iter = host.opts.max_iter;
        ab.warm_in = 1; ab.iters_accumulate = 1; ab.write_u = 1;
        rc = admm_launch(this, ab, st);
        if (rc != CARMPC_OK) return rc;
        pb.idx_list = second_list; pb.count = n_failed; pb.count_dev = nullptr; pb.n_failed = ws_counters + kCntFinal; pb.final_pass = 1;
        rc = polish_launch(this, pb, st);
        if (rc != CARMPC_OK) return rc;
        // whoever is still at "max_iter" is almost always barely infeasible: the dual iterate of its final ADMM state,
        // evaluated exactly, settles it
        if (certify) {
            rc = farkas_decide_launch(this, pb, second_list, n_failed, nullptr, ab.warm, st);
            if (rc != CARMPC_OK) return rc;
            ++k.launches;
        }
        k.launches += 2;
        if (host.opts.polish) {
            // second-pass "infeasible" verdicts need their float64 certificate as well (unverified ones join the fallback)
            CARMPC_CUDA(cudaMemsetAsync(ws_counters + kCntVerify2, 0, sizeof(int), st));
            rc = farkas_verify_launch(this, pb, second_list, n_failed, nullptr, ab.warm, ws_overflow, ws_counters + kCntVerify2, st);
            if (rc != CARMPC_OK) return rc;
            // whatever is still without a proof (no KKT certificate, or out of iterations): float64 fallback
            int handled = 0;
            rc = exact_fallback(this, pb, second_list, n_failed, nullptr, ab.warm, ab.iters, st, &handled);
            if (rc != CARMPC_OK) return rc;
            k.launches += handled > 0 ? 4 : 1;
        }
    }
    if (!r.keep_total) {
        unsigned long long total = 0;
        CARMPC_CUDA(cudaMemcpyAsync(&total, ws_total_iters, sizeof(total), cudaMemcpyDeviceToHost, st));
        CARMPC_CUDA(cudaStreamSynchronize(st));
        k.iters = (int64_t)total;
    }
    last_total_iters = k.iters; last_launches = k.launches;
    return CARMPC_OK;
}

int QPHandle::solve_enqueue(const SolveRequest& r, cudaStream_t st) {
    if (host_only) { set_error("carmpc_qp: this handle was created without a CUDA device; there is no CPU solver"); return CARMPC_ERR_CUDA; }
    if (!host.opts.polish) { set_error("solve_enqueue needs the float64 polish (opts.polish = 1)"); return CARMPC_ERR_INVALID; }
    int rc = ensure_workspace(r.stride);
    if (rc != CARMPC_OK) return rc;
    CARMPC_CUDA(cudaMemsetAsync(ws_counters, 0, sizeof(int) * kCounters, st));
    const int cap = (int)r.count;

    // every stage below (pu, p0, the polish passes, ab, the certificates, the fallback) sees the same disturbance r.c
    PolishBatch pb = polish_batch(*this, r);
    AdmmBatch ab = admm_batch(*this, r);

    // 0. the empty active set (runs near their goal: the unconstrained minimiser is feasible), one thread per run
    PolishBatch pu = pb;
    pu.iters_out = ab.iters;
    rc = polish_unconstrained_launch(this, pu, ws_rest, ws_counters + kCntRest, st);
    if (rc != CARMPC_OK) return rc;
    // 1. the active set certified at the previous step, straight into the float64 polish
    PolishBatch p0 = pb;
    p0.idx_list = ws_rest; p0.count = cap; p0.count_dev = ws_counters + kCntRest;
    p0.rounds = 4; p0.final_pass = 0; p0.n_failed = ws_counters + kCntReuseFailed; p0.failed_list = ws_failed0;
    p0.precheck = 1; p0.Px = admm.Px; p0.Pc = admm.Pc; p0.pre_lo = admm.pre_lo; p0.pre_hi = admm.pre_hi; p0.kpre = admm.kpre;
    p0.iters_out = ab.iters;
    rc = polish_launch(this, p0, st);
    if (rc != CARMPC_OK) return rc;

    // 2. ADMM (warm-started from the previous step's state) for the runs whose set changed, then the polish
    ab.idx_list = ws_failed0; ab.count = cap; ab.count_dev = ws_counters + kCntReuseFailed; ab.narrow = 1;
    rc = admm_launch(this, ab, st);
    if (rc != CARMPC_OK) return rc;
    pb.idx_list = ws_failed0; pb.count = cap; pb.count_dev = ws_counters + kCntReuseFailed;
    rc = polish_launch(this, pb, st);
    if (rc != CARMPC_OK) return rc;
    rc = farkas_verify_launch(this, pb, ws_failed0, cap, ws_counters + kCntReuseFailed, r.warm, ws_failed, ws_counters + kCntFailed, st);
    if (rc != CARMPC_OK) return rc;

    // 3. second pass (tighter) for what is still open, then the float64 fallback: all sized on the device, almost always empty
    ab.idx_list = ws_failed; ab.count_dev = ws_counters + kCntFailed; ab.next = ws_counters + kCntNext2; ab.eps_scale = 0.01f;
    ab.iters_accumulate = 1; ab.write_u = 1;
    rc = admm_launch(this, ab, st);
    if (rc != CARMPC_OK) return rc;
    pb.idx_list = ws_failed; pb.count_dev = ws_counters + kCntFailed; pb.n_failed = ws_counters + kCntFinal; pb.final_pass = 1;
    rc = polish_launch(this, pb, st);
    if (rc != CARMPC_OK) return rc;
    rc = farkas_decide_launch(this, pb, ws_failed, cap, ws_counters + kCntFailed, r.warm, st);
    if (rc != CARMPC_OK) return rc;
    rc = farkas_verify_launch(this, pb, ws_failed, cap, ws_counters + kCntFailed, r.warm, ws_overflow, ws_counters + kCntVerify2, st);
    if (rc != CARMPC_OK) return rc;
    int handled = 0;
    return exact_fallback(this, pb, ws_failed, cap, ws_counters + kCntFailed, r.warm, ab.iters, st, &handled);
}

int QPHandle::solve_seeded(const SolveRequest& r, cudaStream_t st, SolveCounts* counts) {
    if (host_only) { set_error("carmpc_qp: this handle was created without a CUDA device; there is no CPU solver"); return CARMPC_ERR_CUDA; }
    if (!host.opts.polish) { set_error("carmpc_qp_solve with seeds needs the float64 polish (opts.polish = 1)"); return CARMPC_ERR_INVALID; }
    const int64_t batch = r.stride;
    int rc = ensure_workspace(batch);
    if (rc != CARMPC_OK) return rc;
    CARMPC_CUDA(cudaMemsetAsync(ws_polish_stats, 0, sizeof(unsigned long long) * kPolishStats, st));
    CARMPC_CUDA(cudaMemsetAsync(ws_counters + kCntAnchors, 0, sizeof(int) * 2, st));
    CARMPC_CUDA(cudaMemsetAsync(r.status, 0, sizeof(int32_t) * batch, st));     // followers enter the polish as "not infeasible"
    split_seeds_kernel<<<(int)((batch + 255) / 256), 256, 0, st>>>(r.seed, (int)batch, ws_anchor, ws_follow,
                                                                   ws_counters + kCntAnchors, ws_rec_of);
    int n_split[2] = {0, 0};
    CARMPC_CUDA(cudaMemcpyAsync(n_split, ws_counters + kCntAnchors, sizeof(int) * 2, cudaMemcpyDeviceToHost, st));
    CARMPC_CUDA(cudaStreamSynchronize(st));
    SolveRequest part = r;
    part.hold_stats = 1; part.keep_sign = 1;              // the histogram covers anchors and followers
    // multiplier maps of the anchors (1.4 KB each); skipped when there is a per-sample disturbance or too many anchors
    constexpr size_t kRecLam = sizeof(double) * 32 * 5, kRecAct = sizeof(int) * 33;
    if (r.c == nullptr && n_split[0] > 0 && n_split[1] > 0 && (size_t)n_split[0] * (kRecLam + kRecAct) <= ((size_t)1 << 30)) {
        if (n_split[0] > rec_cap) {
            cudaFree(ws_rec_lam); cudaFree(ws_rec_act); ws_rec_lam = nullptr; ws_rec_act = nullptr; rec_cap = 0;
            CARMPC_CUDA(cudaMalloc(&ws_rec_lam, kRecLam * n_split[0]));
            CARMPC_CUDA(cudaMalloc(&ws_rec_act, kRecAct * n_split[0]));
            rec_cap = n_split[0];
        }
        CARMPC_CUDA(cudaMemsetAsync(ws_rec_act, 0xFF, kRecAct * n_split[0], st));      // na = -1: no map yet
        part.records = 1;
    }
    SolveCounts sum, k;
    sum.launches = 1;
    if (n_split[0] > 0) {
        part.idx = ws_anchor; part.count = n_split[0]; part.reuse = 0; part.seed = nullptr;
        rc = solve(part, st, &k);
        if (rc != CARMPC_OK) return rc;
        sum.iters += k.iters; sum.launches += k.launches;
        if (part.records && n_split[1] > 0) {
            rc = farkas_export_launch(this, polish_batch(*this, part), ws_anchor, n_split[0], ws_warm, st);
            if (rc != CARMPC_OK) return rc;
            ++sum.launches;
        }
    }
    if (n_split[1] > 0) {
        part.idx = ws_follow; part.count = n_split[1]; part.reuse = 1; part.seed = r.seed;
        rc = solve(part, st, &k);
        if (rc != CARMPC_OK) return rc;
        sum.iters += k.iters; sum.launches += k.launches; sum.reused = k.reused;
    }
    last_total_iters = sum.iters; last_launches = sum.launches;
    if (counts) *counts = sum;
    return CARMPC_OK;
}

}  // namespace carmpc

using namespace carmpc;

extern "C" {

void carmpc_qp_default_opts(carmpc_qp_opts* o) {
    if (!o) return;
    o->rho = 0.0; o->alpha = 1.8; o->eps_abs = 3e-3; o->eps_rel = 3e-3; o->eps_prim_inf = 1e-4;
    o->max_iter = 4000; o->check_every = 0; o->scaling_iters = 15; o->polish = 1;
}

int carmpc_qp_create(int n, int m, int k, const double* h_H, const double* h_F, const double* h_G, const double* h_Gx,
                     const double* h_Gc, const double* h_lo, const double* h_hi, const double* h_lb,
                     const double* h_ub, const double* h_Px, const double* h_Pc, const double* h_pre_lo,
                     const double* h_pre_hi, const carmpc_qp_opts* opts, void** handle) {
    CARMPC_REQUIRE(handle != nullptr, "handle");
    CARMPC_REQUIRE(n >= 1 && n <= kMaxN, "n must be in [1, 160]");
    CARMPC_REQUIRE(m >= 0 && m <= 1024, "m must be in [0, 1024]");
    CARMPC_REQUIRE(k >= 0 && k <= 64, "k must be in [0, 64]");
    CARMPC_REQUIRE(h_H && h_F && h_lb && h_ub, "null matrix pointer");
    CARMPC_REQUIRE(m == 0 || (h_G && h_Gx && h_lo && h_hi), "null constraint pointer");
    CARMPC_REQUIRE(k == 0 || (h_Px && h_pre_lo && h_pre_hi), "null pre-check pointer");
    carmpc_qp_opts o;
    carmpc_qp_default_opts(&o);
    if (opts) o = *opts;
    if (o.rho <= 0) {
        // automatic penalty: the best fixed rho on the scaled problem falls with the horizon (measured on the
        // region-of-attraction grid: 0.4 / 0.2 / 0.05 / 0.025 for n = 20 / 40 / 80 / 160 variables)
        o.rho = 320.0 / ((double)n * n);
        o.rho = o.rho > 0.4 ? 0.4 : (o.rho < 0.02 ? 0.02 : o.rho);
    }
    // automatic cadence of the convergence checks: a check costs about two plain iterations whatever the problem size, so
    // small problems (cheap iterations) check less often (measured on the config-3 grid: horizon 10 is 8 % faster with 14
    // than with 10, horizon 20 is best at 10)
    if (o.check_every <= 0) o.check_every = n <= 20 ? 14 : 10;
    CARMPC_REQUIRE(o.alpha > 0 && o.alpha < 2, "0 < alpha < 2");
    CARMPC_REQUIRE(o.check_every >= 1 && o.max_iter >= o.check_every, "check_every >= 1, max_iter >= check_every");
    CARMPC_REQUIRE(o.scaling_iters >= 0 && o.scaling_iters <= 100, "scaling_iters");
    QPHandle* q = new QPHandle();
    q->kind = kQP;
    cudaGetDevice(&q->device);
    q->sm = sm_count();
    int rc = qp_host_setup(n, m, k, h_H, h_F, h_G, h_Gx, h_Gc, h_lo, h_hi, h_lb, h_ub, h_Px, h_Pc, h_pre_lo, h_pre_hi, o,
                           &q->host);
    if (rc != CARMPC_OK) { delete q; return rc; }
    QPHost& h = q->host;
    q->admm = h.geo;
    AdmmTables& a = q->admm;
    int n_dev = 0;
    if (cudaGetDeviceCount(&n_dev) != cudaSuccess || n_dev == 0) {
        // no CUDA device: keep the host-side setup inspectable (carmpc_qp_get_setup); every solve fails loudly
        cudaGetLastError();
        q->host_only = true;
        *handle = q;
        return CARMPC_OK;
    }
#define UP(vec, field) do { rc = upload(q, h.vec, &a.field); if (rc != CARMPC_OK) { delete q; return rc; } } while (0)
    UP(P, P); UP(Gs, Gs); UP(GsT, GsT); UP(his, his); UP(Gxs, Gxs); UP(Gcs, Gcs); UP(width, width); UP(Einv_g, Einv_g); UP(Esc_g, Esc_g); UP(Esc_b, Esc_b);
    UP(vpos, vpos); UP(row_id, row_id); UP(lam, lam); UP(lbs, lbs); UP(ubs, ubs); UP(Einv_b, Einv_b); UP(Dinv, Dinv);
    UP(Dsc, Dsc); UP(KF, KF); UP(var_id, var_id); UP(segA, segA); UP(segB, segB); UP(Px, Px); UP(Pc, Pc);
    UP(pre_lo, pre_lo); UP(pre_hi, pre_hi);
#undef UP
    q->tc = h.tc;
    if (h.tc.ok || h.tc_parts.size() > 1) {
        for (const TcPart& part : h.tc_parts) {
            TcTables t = part.t;
            void* d_img = nullptr;
            // chunk images are the sources of cp.async.bulk copies: 16-byte granules (cudaMalloc aligns to 256 bytes)
            if (cudaMalloc(&d_img, part.img.size()) != cudaSuccess) { set_error("cudaMalloc of the tensor-core images failed"); delete q; return CARMPC_ERR_CUDA; }
            q->allocations.push_back(d_img);
            if (cudaMemcpy(d_img, part.img.data(), part.img.size(), cudaMemcpyHostToDevice) != cudaSuccess) { set_error("upload of the tensor-core images failed"); delete q; return CARMPC_ERR_CUDA; }
            t.img = static_cast<const unsigned char*>(d_img);
#define UPT(vec, field) do { rc = upload(q, part.vec, &t.field); if (rc != CARMPC_OK) { delete q; return rc; } } while (0)
            UPT(nwd, nwd); UPT(einv_g, einv_g); UPT(hisf, hisf); UPT(gxsf, gxsf); UPT(gcsf, gcsf);
            UPT(his, his); UPT(gxs, gxs); UPT(gcs, gcs); UPT(row_id, row_id);
            UPT(lam, lam); UPT(lb, lb); UPT(ub, ub); UPT(einv_b, einv_b); UPT(nrl, nrl); UPT(kfv, kfv); UPT(var_id, var_id);
#undef UPT
            q->tc_parts.push_back(t);
        }
        q->tc = q->tc_parts[0];
    }
    PolishTables& p = q->polish;
    p.n = n; p.m = m; p.mt = m + n; p.kpre = k;
#define UP(vec, field) do { rc = upload(q, h.vec, &p.field); if (rc != CARMPC_OK) { delete q; return rc; } } while (0)
    UP(H, H); UP(Hinv, Hinv); UP(F, F); UP(Uu, Uu); UP(AUu, AUu); UP(AH, AH); UP(AHA, AHA); UP(Gx, Gx); UP(Gc, Gc); UP(hi, hi); UP(lo, lo);
    UP(G, G); UP(Eg, Eg); UP(rsign, rsign);
#undef UP
    {
        ExactTables& e = q->exact;
        std::vector<double> GsT((size_t)n * m), lam64(n);
        for (int i = 0; i < m; ++i)
            for (int j = 0; j < n; ++j) GsT[(size_t)j * m + i] = h.Gs64[(size_t)i * n + j];
        for (int j = 0; j < n; ++j) lam64[j] = h.Eb[j] * h.D[j];
#define UPV(vec, field) do { rc = upload(q, vec, &e.field); if (rc != CARMPC_OK) { delete q; return rc; } } while (0)
        // reach of every general row over the input box (single-row Farkas certificates: a row whose bound lies outside
        // [rowmin, rowmax] proves infeasibility by itself)
        std::vector<double> rowmin(m, 0.0), rowmax(m, 0.0), rowabs(m, 0.0);
        for (int i = 0; i < m; ++i)
            for (int j = 0; j < n; ++j) {
                const double g = h.G[(size_t)i * n + j];
                if (g == 0.0) continue;
                const double a = g * h.lo[m + j], b = g * h.hi[m + j];       // box bounds sit behind the general rows
                rowmin[i] += std::min(a, b);
                rowmax[i] += std::max(a, b);
                rowabs[i] += fabs(g) * std::max(fabs(h.lo[m + j]), fabs(h.hi[m + j]));
            }
        UPV(h.Gs64, Gs); UPV(GsT, GsT); UPV(h.Kinv, Kinv); UPV(lam64, lam); UPV(h.Eb, Eb); UPV(h.D, D);
        UPV(rowmin, rowmin); UPV(rowmax, rowmax); UPV(rowabs, rowabs);
#undef UPV
        e.cs = h.cscale; e.rho = o.rho; e.alpha = o.alpha;
    }
    *handle = q;
    return CARMPC_OK;
}

int carmpc_qp_get_setup(void* qp, int which, double* h_out, int capacity) {
    QPHandle* q = check_handle<QPHandle>(qp, kQP);
    CARMPC_REQUIRE(q != nullptr, "not a QP handle");
    const QPHost& h = q->host;
    std::vector<double> tmp;
    const std::vector<double>* src = nullptr;
    switch (which) {
        case 0: src = &h.D; break;
        case 1: src = &h.Eg; break;
        case 2: src = &h.Eb; break;
        case 3: tmp = {h.cscale}; src = &tmp; break;
        case 4: src = &h.Kinv; break;
        case 5: src = &h.Gs64; break;
        case 6: tmp.resize(h.n); for (int j = 0; j < h.n; ++j) tmp[j] = h.Eb[j] * h.D[j]; src = &tmp; break;
        case 7: tmp = {(double)h.samples_per_lane, (double)h.ga_per_warp, (double)h.gb_per_warp, (double)h.mats_in_smem,
                       (double)h.smem_bytes, h.flops_per_iter, h.flops_per_iter_dense, (double)h.geo.ktot,
                       (double)h.geo.m_phys, (double)h.geo.nA_rows}; src = &tmp; break;
        // padded device images, as float64 (tests re-run the kernel's arithmetic on the host from these)
        case 10: tmp.assign(h.P.begin(), h.P.end()); src = &tmp; break;
        case 11: tmp.assign(h.Gs.begin(), h.Gs.end()); src = &tmp; break;
        case 12: tmp.assign(h.GsT.begin(), h.GsT.end()); src = &tmp; break;
        case 13: src = &h.his; break;
        case 14: src = &h.Gxs; break;
        case 15: tmp.assign(h.width.begin(), h.width.end()); src = &tmp; break;
        case 16: tmp.assign(h.vpos.begin(), h.vpos.end()); src = &tmp; break;
        case 17: tmp.assign(h.row_id.begin(), h.row_id.end()); src = &tmp; break;
        case 18: tmp.assign(h.lam.begin(), h.lam.end()); src = &tmp; break;
        case 19: tmp.assign(h.lbs.begin(), h.lbs.end()); src = &tmp; break;
        case 20: tmp.assign(h.ubs.begin(), h.ubs.end()); src = &tmp; break;
        case 21: src = &h.KF; break;
        case 22: tmp.assign(h.var_id.begin(), h.var_id.end()); src = &tmp; break;
        case 23: for (const int4& s4 : h.segA) { tmp.push_back(s4.x); tmp.push_back(s4.y); tmp.push_back(s4.z); tmp.push_back(s4.w); } src = &tmp; break;
        case 24: for (const int2& s2 : h.segB) { tmp.push_back(s2.x); tmp.push_back(s2.y); } src = &tmp; break;
        case 25: tmp.assign(h.Dsc.begin(), h.Dsc.end()); src = &tmp; break;
        case 26: tmp = {(double)h.geo.n, (double)h.geo.m, (double)h.geo.nA_rows, (double)h.geo.m_phys, (double)h.geo.npad4,
                        (double)h.geo.mv4, (double)h.geo.ktot, (double)h.geo.nGA, (double)h.geo.nGB}; src = &tmp; break;
        // tensor-core form (qp_admm_tc.cu): geometry, the chunk images as the float32 words they hold, the per-row tables
        case 30: {
            const TcTables& t = h.tc;
            tmp = {(double)t.ok, (double)t.np, (double)t.mp, (double)t.resident, (double)t.na_stages, (double)t.nb_stages,
                   (double)t.b_stage_bytes, (double)t.smem_bytes};
            for (int p = 0; p < 3; ++p) { tmp.push_back(t.off[p]); tmp.push_back(t.pair_bytes[p]); tmp.push_back(t.nchunks[p]);
                                          tmp.push_back(t.ksteps[p]); tmp.push_back(t.ncols[p]); }
            src = &tmp; break;
        }
        case 31: {
            const std::vector<unsigned char>& img = h.tc_parts[0].img;
            tmp.resize(img.size() / 4);
            for (size_t i = 0; i < tmp.size(); ++i) { float f; memcpy(&f, img.data() + 4 * i, 4); tmp[i] = f; }
            src = &tmp; break;
        }
        case 32: tmp.assign(h.tc_parts[0].nwd.begin(), h.tc_parts[0].nwd.end()); src = &tmp; break;
        case 33: tmp.assign(h.tc_parts[0].einv_g.begin(), h.tc_parts[0].einv_g.end()); src = &tmp; break;
        case 34: src = &h.tc_parts[0].his; break;
        case 35: src = &h.tc_parts[0].gxs; break;
        case 36: src = &h.tc_parts[0].gcs; break;
        case 37: tmp.assign(h.tc_parts[0].row_id.begin(), h.tc_parts[0].row_id.end()); src = &tmp; break;
        case 38: tmp.assign(h.tc_parts[0].lam.begin(), h.tc_parts[0].lam.end()); src = &tmp; break;
        case 39: tmp.assign(h.tc_parts[0].lb.begin(), h.tc_parts[0].lb.end()); src = &tmp; break;
        case 40: tmp.assign(h.tc_parts[0].ub.begin(), h.tc_parts[0].ub.end()); src = &tmp; break;
        case 41: tmp.assign(h.tc_parts[0].einv_b.begin(), h.tc_parts[0].einv_b.end()); src = &tmp; break;
        case 42: tmp.assign(h.tc_parts[0].nrl.begin(), h.tc_parts[0].nrl.end()); src = &tmp; break;
        case 43: src = &h.tc_parts[0].kfv; break;
        default: set_error("carmpc_qp_get_setup: unknown selector %d", which); return CARMPC_ERR_INVALID;
    }
    const int cnt = (int)src->size();
    if (h_out) {
        CARMPC_REQUIRE(capacity >= cnt, "capacity too small");
        memcpy(h_out, src->data(), sizeof(double) * cnt);
    }
    return cnt;
}

int carmpc_qp_solve(void* qp, const double* d_x0, const double* h_xref, const double* d_c, const int32_t* d_seed,
                    int64_t batch, double* d_u0, double* d_objective, int32_t* d_status, int32_t* d_iters, double* d_u_full,
                    float* d_warm, int warm_in, int warm_out, double* d_cert, int64_t* h_seeded, void* stream) {
    QPHandle* q = check_handle<QPHandle>(qp, kQP);
    CARMPC_REQUIRE(q != nullptr, "not a QP handle");
    CARMPC_REQUIRE(batch >= 0 && batch < (int64_t)1 << 31, "batch");
    CARMPC_REQUIRE(h_xref != nullptr, "h_xref");
    CARMPC_REQUIRE(d_warm == nullptr || (d_seed == nullptr && d_cert == nullptr),
                   "d_warm is a starting point of its own: it cannot be combined with d_seed or d_cert");
    CARMPC_REQUIRE(q->host.opts.polish != 0 || (d_seed == nullptr && d_cert == nullptr),
                   "seeds and certificates need the float64 polish (opts.polish = 1)");
    if (h_seeded) *h_seeded = 0;
    if (batch == 0) { q->last_total_iters = 0; q->last_launches = 0; return CARMPC_OK; }
    CARMPC_REQUIRE(d_x0 && d_status, "d_x0 and d_status are required");
    QPBusyGuard guard(q->busy);
    CARMPC_REQUIRE(guard.acquired, "this QP handle is in use by another call (one call per handle at a time)");
    if (q->host_only) { set_error("carmpc_qp: this handle was created without a CUDA device; there is no CPU solver"); return CARMPC_ERR_CUDA; }
    cudaStream_t st = (cudaStream_t)stream;
    const size_t width = (size_t)q->host.m + q->host.n + q->host.kpre;
    if (d_cert) CARMPC_CUDA(cudaMemsetAsync(d_cert, 0, sizeof(double) * width * batch, st));
    SolveRequest r;
    r.x0 = d_x0; r.stride = r.count = batch; r.xref = h_xref; r.c = d_c; r.seed = d_seed;
    r.u0 = d_u0; r.objective = d_objective; r.status = d_status; r.iters = d_iters; r.u_full = d_u_full; r.cert = d_cert;
    r.warm = d_warm; r.warm_in = warm_in; r.warm_out = warm_out;
    if (d_seed == nullptr) return q->solve(r, st);
    SolveCounts k;
    const int rc = q->solve_seeded(r, st, &k);
    if (rc == CARMPC_OK && h_seeded) *h_seeded = k.reused;
    return rc;
}

int carmpc_qp_sensitivity(void* qp, const double* d_x0, const double* d_c, int64_t batch, const int32_t* d_status,
                          const double* d_u_full, const double* d_cert, int rows, double* d_jac, double* d_grad_obj,
                          int32_t* d_flags, void* stream) {
    QPHandle* q = check_handle<QPHandle>(qp, kQP);
    CARMPC_REQUIRE(q != nullptr, "not a QP handle");
    CARMPC_REQUIRE(batch >= 0 && batch < (int64_t)1 << 31, "batch");
    CARMPC_REQUIRE(rows >= 1 && rows <= q->host.n, "1 <= rows <= n");
    CARMPC_REQUIRE(q->host.opts.polish != 0, "sensitivities need the certificates of the float64 polish (opts.polish = 1)");
    if (batch == 0) return CARMPC_OK;
    CARMPC_REQUIRE(d_x0 && d_status && d_u_full && d_cert && d_flags, "d_x0, d_status, d_u_full, d_cert and d_flags are required");
    if (q->host_only) { set_error("carmpc_qp: this handle was created without a CUDA device; there is no CPU solver"); return CARMPC_ERR_CUDA; }
    // reads only the handle's constant tables: no workspace, so no busy guard is needed
    return sensitivity_launch(q, d_x0, d_c, batch, d_status, d_u_full, d_cert, rows, d_jac, d_grad_obj, d_flags,
                              (cudaStream_t)stream);
}

int carmpc_qp_solve_host(void* qp, const double* h_x0, const double* h_xref, const double* h_c, int64_t batch,
                         double* h_u0, double* h_objective, int32_t* h_status, int32_t* h_iters, double* h_u_full) {
    QPHandle* q = check_handle<QPHandle>(qp, kQP);
    CARMPC_REQUIRE(q != nullptr, "not a QP handle");
    CARMPC_REQUIRE(batch >= 0 && batch < (int64_t)1 << 31, "batch");
    if (batch == 0) return CARMPC_OK;
    CARMPC_REQUIRE(h_x0 && h_xref && h_status, "null host pointer");
    if (q->host_only) { set_error("carmpc_qp: this handle was created without a CUDA device; there is no CPU solver"); return CARMPC_ERR_CUDA; }
    QPBusyGuard guard(q->busy);
    CARMPC_REQUIRE(guard.acquired, "this QP handle is in use by another call (one call per handle at a time)");
    int rc = q->ensure_io(batch, h_u_full != nullptr);
    if (rc != CARMPC_OK) return rc;
    cudaStream_t st = nullptr;
    // states arrive as the reference passes them (batch x 4, row-major): one copy, re-laid out to SoA on the device
    CARMPC_CUDA(cudaMemcpyAsync(q->io_x0_aos, h_x0, sizeof(double) * 4 * batch, cudaMemcpyHostToDevice, st));
    aos_to_soa_kernel<<<(int)((batch + 255) / 256), 256, 0, st>>>(q->io_x0_aos, q->io_x0, batch, 4);
    if (h_c) CARMPC_CUDA(cudaMemcpyAsync(q->io_c, h_c, sizeof(double) * batch, cudaMemcpyHostToDevice, st));
    SolveRequest r;
    r.x0 = q->io_x0; r.stride = r.count = batch; r.xref = h_xref; r.c = h_c ? q->io_c : nullptr;
    r.u0 = q->io_u0; r.objective = q->io_obj; r.status = q->io_status; r.iters = q->io_iters;
    r.u_full = h_u_full ? q->io_full : nullptr;
    rc = q->solve(r, st);
    if (rc != CARMPC_OK) return rc;
    return download(q, batch, h_u0, h_objective, h_status, h_iters, h_u_full, st);
}

int carmpc_qp_map_host(void* qp, const double* h_axes, const int32_t dims[4], const int32_t axis_to_state[4],
                       const int32_t block[4], const double* h_xref, double* h_u0, double* h_objective, int32_t* h_status,
                       int32_t* h_iters, int64_t* h_seeded) {
    QPHandle* q = check_handle<QPHandle>(qp, kQP);
    CARMPC_REQUIRE(q != nullptr, "not a QP handle");
    CARMPC_REQUIRE(h_axes && dims && axis_to_state && h_xref && h_status, "null pointer");
    if (q->host_only) { set_error("carmpc_qp: this handle was created without a CUDA device; there is no CPU solver"); return CARMPC_ERR_CUDA; }
    MapGrid g;
    int64_t n = 1;
    int off = 0, seen = 0;
    bool blocked = false;
    for (int k = 0; k < 4; ++k) {
        CARMPC_REQUIRE(dims[k] >= 1 && dims[k] <= 4096, "each axis must have 1..4096 points");
        CARMPC_REQUIRE(axis_to_state[k] >= 0 && axis_to_state[k] < 4, "axis_to_state entries must be 0..3");
        CARMPC_REQUIRE(block == nullptr || block[k] >= 1, "block entries must be >= 1");
        seen |= 1 << axis_to_state[k];
        g.dims[k] = dims[k]; g.state_of_axis[k] = axis_to_state[k]; g.offset[k] = off;
        g.block[k] = block ? block[k] : 1;
        blocked = blocked || g.block[k] > 1;
        off += dims[k];
        n *= dims[k];
    }
    CARMPC_REQUIRE(seen == 15, "axis_to_state must be a permutation of 0..3");
    CARMPC_REQUIRE(n < (int64_t)1 << 31, "grid too large for one call");
    if (h_seeded) *h_seeded = 0;
    QPBusyGuard guard(q->busy);
    CARMPC_REQUIRE(guard.acquired, "this QP handle is in use by another call (one call per handle at a time)");
    int rc = q->ensure_io(n, false);
    if (rc != CARMPC_OK) return rc;
    if (q->io_axes == nullptr) CARMPC_CUDA(cudaMalloc(&q->io_axes, sizeof(double) * 4 * 4096));
    cudaStream_t st = nullptr;
    CARMPC_CUDA(cudaMemcpyAsync(q->io_axes, h_axes, sizeof(double) * off, cudaMemcpyHostToDevice, st));
    map_expand_kernel<<<(int)((n + 255) / 256), 256, 0, st>>>(q->io_axes, g, n, q->io_x0, q->io_seed);
    CARMPC_CUDA(cudaGetLastError());
    SolveRequest r;
    r.x0 = q->io_x0; r.stride = r.count = n; r.xref = h_xref;
    r.u0 = h_u0 ? q->io_u0 : nullptr; r.objective = h_objective ? q->io_obj : nullptr; r.status = q->io_status; r.iters = q->io_iters;
    if (blocked && q->host.opts.polish) {
        r.seed = q->io_seed;
        SolveCounts k;
        rc = q->solve_seeded(r, st, &k);
        if (rc == CARMPC_OK && h_seeded) *h_seeded = k.reused;
    } else {
        rc = q->solve(r, st);
    }
    if (rc != CARMPC_OK) return rc;
    return download(q, n, h_u0, h_objective, h_status, h_iters, nullptr, st);
}

int carmpc_qp_polish_stats(void* qp, int64_t* h_hist20) {
    QPHandle* q = check_handle<QPHandle>(qp, kQP);
    CARMPC_REQUIRE(q != nullptr, "not a QP handle");
    CARMPC_REQUIRE(h_hist20 != nullptr, "h_hist20");
    for (int i = 0; i < kPolishStats; ++i) h_hist20[i] = 0;
    if (q->ws_polish_stats == nullptr) return CARMPC_OK;
    unsigned long long tmp[kPolishStats];
    CARMPC_CUDA(cudaMemcpy(tmp, q->ws_polish_stats, sizeof(tmp), cudaMemcpyDeviceToHost));
    for (int i = 0; i < kPolishStats; ++i) h_hist20[i] = (int64_t)tmp[i];
    return CARMPC_OK;
}

int carmpc_qp_tensor_mode(void* qp, int mode, int64_t* h_info) {
    QPHandle* q = check_handle<QPHandle>(qp, kQP);
    CARMPC_REQUIRE(q != nullptr, "not a QP handle");
    CARMPC_REQUIRE(mode <= 3, "mode must be 0, 1, 2, 3 or negative (query)");
    if (mode >= 0) q->tensor_mode = mode;
    if (h_info) {
        for (int i = 0; i < 16; ++i) h_info[i] = 0;
        h_info[0] = q->tensor_mode; h_info[1] = q->tc_parts.empty() ? 0 : (int64_t)q->tc_parts.size();
        h_info[2] = q->last_tc_samples; h_info[3] = q->tc.resident;
        if (q->ws_prof != nullptr) {
            unsigned long long tmp[16];
            CARMPC_CUDA(cudaMemcpy(tmp, q->ws_prof, sizeof(tmp), cudaMemcpyDeviceToHost));
            for (int i = 0; i < 12; ++i) h_info[4 + i] = (int64_t)tmp[i];
            // (h_info has 16 slots: counters 0..11)
        }
    }
    return CARMPC_OK;
}

int carmpc_qp_last_stats(void* qp, int64_t* h_total_iters, int64_t* h_launches) {
    QPHandle* q = check_handle<QPHandle>(qp, kQP);
    CARMPC_REQUIRE(q != nullptr, "not a QP handle");
    if (h_total_iters) *h_total_iters = q->last_total_iters;
    if (h_launches) *h_launches = q->last_launches;
    return CARMPC_OK;
}

}  // extern "C"
