// Monte-Carlo closed loops: very many independent runs of  plant step -> (observer) -> MPC QP  in lock-step.
//
// Order of operations is the reference's loop (examples/run_MPCOutputFB.py:29-41, run_MPCStateFB.py:29-39): the plant
// (lib/simulator.py:51-69, forward Euler of the kinematic bicycle) moves first with the previous input ([0, 0] at the
// first step), then the controller steps on the new output: Luenberger observer (lib/mpc.py:448) for output feedback,
// the state itself for state feedback, then one condensed QP per run (lib/mpc.py:461-478 / :318-335).  A run whose QP is
// infeasible stops there, as the reference raises OutsideTheRegionOfAttractionError.
//
// The disturbance mode (mode 2) is the controller for constant disturbances
// (MPCOutputFBWithDisturbance): the plant gets a constant per-run disturbance d_r after its Euler step (Bd_p d_r) and in
// its output (Cd_p d_r); the augmented observer keeps a scalar estimate d^ beside x^,
//     i = y - C x^ - Cd d^ ,   x^' = A x^ + Bd d^ + B u_prev + L1 i ,   d^' = d^ + L2 . i ,
// and the QP of the run takes d^' as its disturbance c (bounds shifted by Gc c).  The d^ buffer itself is the c array
// the QP stages read, so its address is fixed across steps and the captured step graph stays valid.
//
// One thread per run for plant + observer (4 state and 2 input registers); the QPs of all live runs go through the
// batched solver with the previous step's ADMM state as warm start.
//
// Noise and monitor (any mode): process noise Lw z_w is added to the plant state after
// the Euler step (and after Bd_p d_r), the state is then checked against the caller's rows [a | b] with the membership
// chain of K1 (a violation never stops a run), and measurement noise Lv z_v enters what the controller sees.  z_w, z_v
// are four standard normals each from Philox4x64-10 (philox.cuh) at counter (first_run + run, step, 0 / 1, 0), key
// (seed, 0): they depend on nothing but the global run id and the step, so warm-start mode, graph replay and batch
// composition draw the same noise.  Both are compile-time switches of loop_advance_kernel: with both off it has none of
// their code.
//
// Goal (any mode): the caller's goal rows [a | b] are checked on the same true plant state as the monitor, with the same
// chain.  The run still solves its QP at that step, so a QP that is not solved stops the run as a failure first (the
// reference raises before it tests the goal); a solved QP with the state inside stops the run as arrived: its input is
// not applied and it is never moved, solved or counted again.  The verdict of the rows waits for the QP's in a loop-owned
// byte per run.  A third compile-time switch of loop_advance_kernel and loop_apply_kernel: with it off both are the
// kernels without a goal.
#include <math.h>
#include <string.h>

#include <stdlib.h>

#include "philox.cuh"
#include "qp_internal.cuh"

namespace carmpc {

namespace {

struct LoopConst {
    double A[16], B[8], C[12], L[12];
    double Bd[4], Cd[3], L2[3], Bdp[4], Cdp[3];     // mode 2: disturbance model, its observer gain, how d_r enters the plant
    double dt, l1;
    int mode;            // 0 state feedback, 1 output feedback, 2 output feedback with a disturbance estimate
};

// Noise factors of a call (carmpc_loop_noise): v = Lv z, w = Lw z, row-major 4 x 4.
struct LoopNoise {
    uint64_t seed;
    int64_t first_run;
    double Lw[16], Lv[16];
};

// A monitor's or a goal's row set on the device (carmpc_loop_rows): the rows in a loop-owned copy, rows x 5, and the
// outputs.
struct LoopRows {
    const double* Ab;
    int rows;
    int32_t* step;                  // runs: monitor - first step whose state violates a row; goal - arrival step; -1 none
    int32_t* row;                   // runs (monitor only, nullable): lowest violated row at that step, -1 none
    int32_t* per_step;              // steps (nullable): runs violating / arriving at the step
};

// K1's mode-0 chain: the first row the state violates, -1 none.  A NaN never satisfies <=.
__device__ __forceinline__ int first_violated(const LoopRows& R, const double s[4]) {
    for (int r = 0; r < R.rows; ++r) {
        const double* a = R.Ab + 5 * r;
        const double lhs = fma(__ldg(a + 3), s[3], fma(__ldg(a + 2), s[2], fma(__ldg(a + 1), s[1], __ldg(a) * s[0])));
        if (!(lhs <= __ldg(a + 4))) return r;
    }
    return -1;
}

// per_step[step] += the threads with hit, one atomic per warp (and per group of threads that arrive together)
__device__ __forceinline__ void count_per_warp(int32_t* per_step, int step, bool hit) {
    const unsigned act = __activemask();
    const unsigned h = __ballot_sync(act, hit);
    if (h != 0 && (int)(threadIdx.x & 31) == __ffs(act) - 1) atomicAdd(per_step + step, __popc(h));
}

// plant step with the previous input, observer update, estimate -> QP input; builds the list of live runs.
// kNoise / kMonitor / kGoal: process and measurement noise, monitor rows, goal rows; step is the step number of
// host-driven steps.  kGoal: inside (loop-owned, runs) keeps whether the state of this step is inside the goal until
// loop_apply_kernel knows its QP.
template <bool kNoise, bool kMonitor, bool kGoal>
__global__ void __launch_bounds__(256)
loop_advance_kernel(const LoopConst K, int64_t runs, double* __restrict__ x, double* __restrict__ xhat,
                    const double* __restrict__ u_prev, const int32_t* __restrict__ fail_step,
                    double* __restrict__ est, int* __restrict__ live_list, int* __restrict__ live_count,
                    double* __restrict__ traj_step, const int* __restrict__ step_dev,
                    double* __restrict__ dhat, const double* __restrict__ d_plant, const LoopNoise N,
                    const LoopRows M, int step, const LoopRows G, uint8_t* inside) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= runs) return;
    // replayed steps (CUDA graph) read the step number on the device: traj_step is then the base of the trajectory
    if (traj_step != nullptr && step_dev != nullptr) traj_step += (size_t)*step_dev * 4 * runs;
    if ((kNoise || kMonitor) && step_dev != nullptr) step = *step_dev;
    bool viol = false;
    double s[4], u[2];
#pragma unroll
    for (int c = 0; c < 4; ++c) s[c] = x[c * runs + i];
    const bool alive = fail_step[i] < 0 && (!kGoal || G.step[i] < 0);
    if (alive) {
        u[0] = u_prev[i];
        u[1] = u_prev[runs + i];
        // state + dt * [v cos(psi), v sin(psi), v / l1 * tan(delta), a]      (rate * dt + state, as the reference)
        const double psi = s[2], v = s[3];
        const double r0 = v * cos(psi), r1 = v * sin(psi), r2 = v / K.l1 * tan(u[1]), r3 = u[0];
        s[0] = r0 * K.dt + s[0];
        s[1] = r1 * K.dt + s[1];
        s[2] = r2 * K.dt + s[2];
        s[3] = r3 * K.dt + s[3];
        double dr = 0.0;
        if (K.mode == 2) {
            // the run's true constant disturbance, added after the Euler step (component-wise)
            if (d_plant != nullptr) dr = d_plant[i];
#pragma unroll
            for (int c = 0; c < 4; ++c) s[c] = s[c] + K.Bdp[c] * dr;
        }
        double vm[4] = {0.0, 0.0, 0.0, 0.0};      // measurement noise
        if (kNoise) {
            const uint64_t run = (uint64_t)(N.first_run + i);
            double z[4];
            normal4(N.seed, run, (uint64_t)step, 0, z);
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                double w = 0.0;
#pragma unroll
                for (int j = 0; j < 4; ++j) w += N.Lw[c * 4 + j] * z[j];
                s[c] = s[c] + w;
            }
            normal4(N.seed, run, (uint64_t)step, 1, z);
#pragma unroll
            for (int c = 0; c < 4; ++c) {
#pragma unroll
                for (int j = 0; j < 4; ++j) vm[c] += N.Lv[c * 4 + j] * z[j];
            }
        }
#pragma unroll
        for (int c = 0; c < 4; ++c) x[c * runs + i] = s[c];
        if (kMonitor) {
            // a non-finite state violates the first row
            const int bad = first_violated(M, s);
            viol = bad >= 0;
            if (viol) {
                if (M.step != nullptr && M.step[i] < 0) M.step[i] = step;
                if (M.row != nullptr && M.row[i] < 0) M.row[i] = bad;
            }
        }
        // a non-finite state is never inside (an infinite coordinate may satisfy a row)
        if (kGoal)
            inside[i] = isfinite(s[0]) && isfinite(s[1]) && isfinite(s[2]) && isfinite(s[3]) && first_violated(G, s) == -1;
        double e[4];
        if (K.mode == 2) {
            // augmented observer: y = C s + Cd_p d_r measured, innovation against C x^ + Cd d^
            double xh[4], innov[3];
            const double dh = dhat[i];
#pragma unroll
            for (int c = 0; c < 4; ++c) xh[c] = xhat[c * runs + i];
#pragma unroll
            for (int r = 0; r < 3; ++r) {
                double y = K.Cdp[r] * dr, yh = K.Cd[r] * dh;
#pragma unroll
                for (int c = 0; c < 4; ++c) { y += K.C[r * 4 + c] * s[c]; yh += K.C[r * 4 + c] * xh[c]; }
                if (kNoise) y += vm[r];
                innov[r] = y - yh;
            }
            double dn = dh;
#pragma unroll
            for (int r = 0; r < 4; ++r) {
                double t = K.Bd[r] * dh;
#pragma unroll
                for (int c = 0; c < 4; ++c) t += K.A[r * 4 + c] * xh[c];
                t += K.B[r * 2 + 0] * u[0] + K.B[r * 2 + 1] * u[1];
#pragma unroll
                for (int c = 0; c < 3; ++c) t += K.L[r * 3 + c] * innov[c];
                e[r] = t;
            }
#pragma unroll
            for (int c = 0; c < 3; ++c) dn += K.L2[c] * innov[c];
#pragma unroll
            for (int c = 0; c < 4; ++c) xhat[c * runs + i] = e[c];
            dhat[i] = dn;                  // = the QP's disturbance c of this run
        } else if (K.mode == 1) {
            double xh[4], innov[3];
#pragma unroll
            for (int c = 0; c < 4; ++c) xh[c] = xhat[c * runs + i];
#pragma unroll
            for (int r = 0; r < 3; ++r) {
                double y = 0, yh = 0;
#pragma unroll
                for (int c = 0; c < 4; ++c) { y += K.C[r * 4 + c] * s[c]; yh += K.C[r * 4 + c] * xh[c]; }
                if (kNoise) y += vm[r];
                innov[r] = y - yh;
            }
#pragma unroll
            for (int r = 0; r < 4; ++r) {
                double t = 0;
#pragma unroll
                for (int c = 0; c < 4; ++c) t += K.A[r * 4 + c] * xh[c];
                t += K.B[r * 2 + 0] * u[0] + K.B[r * 2 + 1] * u[1];
#pragma unroll
                for (int c = 0; c < 3; ++c) t += K.L[r * 3 + c] * innov[c];
                e[r] = t;
            }
#pragma unroll
            for (int c = 0; c < 4; ++c) xhat[c * runs + i] = e[c];
        } else {
#pragma unroll
            for (int c = 0; c < 4; ++c) e[c] = kNoise ? s[c] + vm[c] : s[c];
        }
#pragma unroll
        for (int c = 0; c < 4; ++c) est[c * runs + i] = e[c];
        live_list[atomicAdd(live_count, 1)] = (int)i;
    }
    if (kMonitor && M.per_step != nullptr) count_per_warp(M.per_step, step, viol);
    if (traj_step != nullptr) {
#pragma unroll
        for (int c = 0; c < 4; ++c) traj_step[c * runs + i] = s[c];
    }
}

// take the QP results of the live runs: new input, or mark the run as failed at this step; kGoal: a solved run whose state
// was inside the goal arrives instead of taking its input
template <bool kGoal>
__global__ void __launch_bounds__(256)
loop_apply_kernel(int64_t runs, int step, const int* __restrict__ live_list, int live, const int* __restrict__ live_dev,
                  const double* __restrict__ u0, const int32_t* __restrict__ status, double* __restrict__ u_prev,
                  int32_t* __restrict__ fail_step, const int* __restrict__ step_dev, const LoopRows G,
                  const uint8_t* inside) {
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (live_dev != nullptr) live = min(live, *live_dev);
    if (step_dev != nullptr) step = *step_dev;
    if (q >= live) return;
    const int i = live_list[q];
    bool arrived = false;
    if (status[i] == CARMPC_QP_SOLVED) {
        if (kGoal && inside[i]) {
            G.step[i] = step;
            arrived = true;
        } else {
            u_prev[i] = u0[i];
            u_prev[runs + i] = u0[runs + i];
        }
    } else {
        fail_step[i] = step;
    }
    if (kGoal && G.per_step != nullptr) count_per_warp(G.per_step, step, arrived);
}

// replayed steps: the input (and disturbance-estimate) logs of this step, then the step number moves on (one thread, after
// everything that read it)
__global__ void __launch_bounds__(256)
loop_log_kernel(int64_t runs, const double* __restrict__ u_prev, double* __restrict__ u_log, const double* __restrict__ dhat,
                double* __restrict__ dhat_log, const int* __restrict__ step_dev) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= 2 * runs) return;
    if (u_log != nullptr) u_log[(size_t)*step_dev * 2 * runs + i] = u_prev[i];
    if (dhat_log != nullptr && i < runs) dhat_log[(size_t)*step_dev * runs + i] = dhat[i];
}
__global__ void loop_next_kernel(int* step_dev) { *step_dev += 1; }
__global__ void loop_set_kernel(int* step_dev, int v) { *step_dev = v; }

__global__ void fill_i32(int32_t* p, int64_t n, int32_t v) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) p[i] = v;
}

template <bool kNoise, bool kMonitor>
auto advance_variant(bool goal) {
    return goal ? loop_advance_kernel<kNoise, kMonitor, true> : loop_advance_kernel<kNoise, kMonitor, false>;
}

// Mode-2 state and logs of a run set (all nullable: d^ starts at 0, d_r is 0, d^ is kept in a buffer of the driver).
struct LoopDisturbance {
    const double* dhat_init;
    const double* d_plant;
    double* dhat_final;
    double* dhat_log;
};

// The device side of a row set (h == nullptr: none, *d all null): the rows copied into the loop-owned buffer *Ab, the step
// and row outputs set to -1, the per-step count to 0.
cudaError_t rows_to_device(const carmpc_loop_rows* h, int64_t runs, int steps, cudaStream_t st, double** Ab, LoopRows* d) {
    *d = {nullptr, 0, nullptr, nullptr, nullptr};
    if (h == nullptr) return cudaSuccess;
    cudaError_t e = cudaMalloc(Ab, sizeof(double) * 5 * h->rows);
    if (e == cudaSuccess) e = cudaMemcpyAsync(*Ab, h->h_Ab, sizeof(double) * 5 * h->rows, cudaMemcpyHostToDevice, st);
    if (e != cudaSuccess) return e;
    const int blocks = (int)((runs + 255) / 256);
    if (h->d_step) fill_i32<<<blocks, 256, 0, st>>>(h->d_step, runs, -1);
    if (h->d_row) fill_i32<<<blocks, 256, 0, st>>>(h->d_row, runs, -1);
    if (h->d_per_step && steps > 0) e = cudaMemsetAsync(h->d_per_step, 0, sizeof(int32_t) * steps, st);
    *d = {*Ab, h->rows, h->d_step, h->d_row, h->d_per_step};
    return e;
}

// The loop shared by every mode: host-driven first steps, then one captured CUDA graph with the step number on the device.
int closed_loop_run(QPHandle* q, const LoopConst& K, const double* h_xref, int steps, int warm_start, const double* d_x_init,
                    const double* d_xhat_init, int64_t runs, double* d_final, int32_t* d_fail_step, double* d_traj,
                    double* d_u_log, const LoopDisturbance& D, const carmpc_loop_noise* noise,
                    const carmpc_loop_rows* monitor, const carmpc_loop_rows* goal, int64_t* h_total_iters, void* stream) {
    if (q->host_only) { set_error("carmpc_closed_loop: this QP handle was created without a CUDA device"); return CARMPC_ERR_CUDA; }
    QPBusyGuard guard(q->busy);
    CARMPC_REQUIRE(guard.acquired, "this QP handle is in use by another call (one call per handle at a time)");
    const bool dist = K.mode == 2;
    // The loop runs on its own (capturable) stream, ordered after the caller's stream by an event and joined at the end by
    // the final synchronisation: the legacy default stream cannot be captured into a graph.
    cudaStream_t user_st = (cudaStream_t)stream, st = nullptr;
    cudaEvent_t ev = nullptr;
    bool graph_ok = cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking) == cudaSuccess &&
                    cudaEventCreateWithFlags(&ev, cudaEventDisableTiming) == cudaSuccess;
    if (graph_ok) graph_ok = cudaEventRecord(ev, user_st) == cudaSuccess && cudaStreamWaitEvent(st, ev, 0) == cudaSuccess;
    if (!graph_ok) { cudaGetLastError(); if (st) cudaStreamDestroy(st); st = user_st; }

    const int mt = q->admm.mt;
    double *x = d_final, *xhat = nullptr, *est = nullptr, *u_prev = nullptr, *u0 = nullptr, *dhat_own = nullptr;
    int32_t* status = nullptr;
    int *live_list = nullptr, *live_count = nullptr;
    float* warm = nullptr;
    double *monitor_Ab = nullptr, *goal_Ab = nullptr;
    uint8_t* inside = nullptr;
    int rc = CARMPC_OK;
    auto cleanup = [&]() { if (st != user_st) { cudaStreamSynchronize(st); cudaStreamDestroy(st); } if (ev) cudaEventDestroy(ev);
                           cudaFree(xhat); cudaFree(est); cudaFree(u_prev); cudaFree(u0); cudaFree(status); cudaFree(live_list);
                           cudaFree(live_count); cudaFree(warm); cudaFree(dhat_own); cudaFree(monitor_Ab);
                           cudaFree(goal_Ab); cudaFree(inside); };
#define TRY(call) do { cudaError_t e__ = (call); if (e__ != cudaSuccess) { set_error("%s: %s", #call, cudaGetErrorString(e__)); cleanup(); return CARMPC_ERR_CUDA; } } while (0)
    TRY(cudaMalloc(&xhat, sizeof(double) * 4 * runs));
    TRY(cudaMalloc(&est, sizeof(double) * 4 * runs));
    TRY(cudaMalloc(&u_prev, sizeof(double) * 2 * runs));
    TRY(cudaMalloc(&u0, sizeof(double) * 2 * runs));
    TRY(cudaMalloc(&status, sizeof(int32_t) * runs));
    TRY(cudaMalloc(&live_list, sizeof(int) * runs));
    TRY(cudaMalloc(&live_count, sizeof(int) * 2));      // [0] live runs of the step, [1] step number of replayed steps
    if (warm_start) TRY(cudaMalloc(&warm, sizeof(float) * (size_t)mt * runs));
    // mode 2: the disturbance estimate of every run, which is also the QP's per-run c (fixed address: graph-safe)
    double* dhat = nullptr;
    if (dist) {
        dhat = D.dhat_final;
        if (dhat == nullptr) { TRY(cudaMalloc(&dhat_own, sizeof(double) * runs)); dhat = dhat_own; }
        if (D.dhat_init != nullptr) {
            if (D.dhat_init != dhat) TRY(cudaMemcpyAsync(dhat, D.dhat_init, sizeof(double) * runs, cudaMemcpyDeviceToDevice, st));
        } else {
            TRY(cudaMemsetAsync(dhat, 0, sizeof(double) * runs, st));
        }
    }
    const double* c_qp = dhat;
    if (x != d_x_init) TRY(cudaMemcpyAsync(x, d_x_init, sizeof(double) * 4 * runs, cudaMemcpyDeviceToDevice, st));
    TRY(cudaMemcpyAsync(xhat, d_xhat_init ? d_xhat_init : d_x_init, sizeof(double) * 4 * runs, cudaMemcpyDeviceToDevice, st));
    TRY(cudaMemsetAsync(u_prev, 0, sizeof(double) * 2 * runs, st));
    const int blocks = (int)((runs + 255) / 256);
    fill_i32<<<blocks, 256, 0, st>>>(d_fail_step, runs, -1);
    // noise, monitor and goal: kernel arguments by value (a captured graph keeps them); the rows and the goal's pending
    // verdict in buffers the loop owns, fixed addresses like every other buffer of the step
    LoopNoise nz;
    memset(&nz, 0, sizeof(nz));
    if (noise != nullptr) {
        nz.seed = noise->seed;
        nz.first_run = noise->first_run;
        memcpy(nz.Lw, noise->Lw, sizeof(nz.Lw));
        memcpy(nz.Lv, noise->Lv, sizeof(nz.Lv));
    }
    LoopRows mon, gl;
    TRY(rows_to_device(monitor, runs, steps, st, &monitor_Ab, &mon));
    TRY(rows_to_device(goal, runs, steps, st, &goal_Ab, &gl));
    if (goal != nullptr) {
        TRY(cudaMalloc(&inside, runs));
        TRY(cudaMemsetAsync(inside, 0, runs, st));
    }
    const bool with_noise = noise != nullptr, with_monitor = monitor != nullptr, with_goal = goal != nullptr;
    auto advance = [&](int k, double* traj_step, const int* step_dev) {
        auto kern = with_noise ? (with_monitor ? advance_variant<true, true>(with_goal) : advance_variant<true, false>(with_goal))
                               : (with_monitor ? advance_variant<false, true>(with_goal) : advance_variant<false, false>(with_goal));
        kern<<<blocks, 256, 0, st>>>(K, runs, x, xhat, u_prev, d_fail_step, est, live_list, live_count, traj_step, step_dev,
                                     dhat, D.d_plant, nz, mon, k, gl, inside);
    };
    auto apply = with_goal ? loop_apply_kernel<true> : loop_apply_kernel<false>;
    int64_t total_iters = 0;
    bool warm_valid = false;
    // the iteration total accumulates on the device over the steps (one read at the end instead of one per step)
    rc = q->ensure_workspace(runs);
    if (rc != CARMPC_OK) { cleanup(); return rc; }
    TRY(cudaMemsetAsync(q->ws_total_iters, 0, sizeof(unsigned long long), st));
    // the QP of every step: the live runs (est, indexed like the runs), warm-started once a step has run
    SolveRequest req;
    req.x0 = est; req.stride = runs; req.xref = h_xref; req.c = c_qp; req.idx = live_list;
    req.u0 = u0; req.status = status; req.warm = warm; req.warm_out = warm ? 1 : 0; req.keep_total = 1;
    req.certify_shifted = dist ? 1 : 0;       // host-driven steps certify on the disturbance-shifted bounds too
    // One enqueue-only step (every count stays on the device).  step_dev == nullptr: the step number k comes from the host.
    auto enqueue_step = [&](int k, const int* step_dev) -> int {
        cudaError_t e = cudaMemsetAsync(live_count, 0, sizeof(int), st);
        if (e != cudaSuccess) { set_error("cudaMemsetAsync: %s", cudaGetErrorString(e)); return CARMPC_ERR_CUDA; }
        advance(k, d_traj ? (step_dev ? d_traj : d_traj + (size_t)k * 4 * runs) : nullptr, step_dev);
        SolveRequest r = req;
        r.count = runs; r.count_dev = live_count; r.warm_in = 1;
        const int rc2 = q->solve_enqueue(r, st);
        if (rc2 != CARMPC_OK) return rc2;
        apply<<<blocks, 256, 0, st>>>(runs, k, live_list, (int)runs, live_count, u0, status, u_prev, d_fail_step, step_dev, gl, inside);
        if (step_dev) {
            if (d_u_log || D.dhat_log)
                loop_log_kernel<<<(int)((2 * runs + 255) / 256), 256, 0, st>>>(runs, u_prev, d_u_log, dhat, D.dhat_log, step_dev);
        } else {
            if (d_u_log) e = cudaMemcpyAsync(d_u_log + (size_t)k * 2 * runs, u_prev, sizeof(double) * 2 * runs, cudaMemcpyDeviceToDevice, st);
            if (e == cudaSuccess && D.dhat_log)
                e = cudaMemcpyAsync(D.dhat_log + (size_t)k * runs, dhat, sizeof(double) * runs, cudaMemcpyDeviceToDevice, st);
            if (e != cudaSuccess) { set_error("cudaMemcpyAsync: %s", cudaGetErrorString(e)); return CARMPC_ERR_CUDA; }
        }
        if (step_dev) loop_next_kernel<<<1, 1, 0, st>>>(live_count + 1);
        return CARMPC_OK;
    };
    for (int k = 0; k < steps; ++k) {
        if (warm_valid && warm_start != 2) {
            // Every later step only enqueues: the number of live runs, of runs whose active set changed, of second-pass and
            // fallback samples all stay on the device (kernels sized for the upper bound read them there), so the steps
            // run back to back on the GPU without a host round trip.  The first such step is launched kernel by kernel
            // (it also fills the kernel-attribute caches); the remaining ones are ONE captured CUDA graph replayed with
            // the step number on the device, so that a slow host (thousands of small launches otherwise) cannot stretch
            // the loop.
            if (!graph_ok || k + 2 >= steps || k < 2) {
                rc = enqueue_step(k, nullptr);
                if (rc != CARMPC_OK) { cleanup(); return rc; }
                continue;
            }
            cudaGraph_t graph = nullptr;
            cudaGraphExec_t exec = nullptr;
            loop_set_kernel<<<1, 1, 0, st>>>(live_count + 1, k);
            if (cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal) != cudaSuccess) {
                // no capture possible here (e.g. the caller is capturing itself): launch the steps one by one
                cudaGetLastError();
                graph_ok = false;
                rc = enqueue_step(k, nullptr);
                if (rc != CARMPC_OK) { cleanup(); return rc; }
                continue;
            }
            rc = enqueue_step(k, live_count + 1);
            cudaError_t ce = cudaStreamEndCapture(st, &graph);
            if (rc == CARMPC_OK && ce != cudaSuccess) { set_error("cudaStreamEndCapture: %s", cudaGetErrorString(ce)); rc = CARMPC_ERR_CUDA; }
            if (rc == CARMPC_OK && cudaGraphInstantiate(&exec, graph, 0) != cudaSuccess) { set_error("cudaGraphInstantiate failed"); rc = CARMPC_ERR_CUDA; }
            for (; rc == CARMPC_OK && k < steps; ++k)
                if (cudaGraphLaunch(exec, st) != cudaSuccess) { set_error("cudaGraphLaunch failed"); rc = CARMPC_ERR_CUDA; }
            if (exec) cudaGraphExecDestroy(exec);
            if (graph) cudaGraphDestroy(graph);
            if (rc != CARMPC_OK) { cudaGetLastError(); cleanup(); return rc; }
            break;
        }
        TRY(cudaMemsetAsync(live_count, 0, sizeof(int), st));
        advance(k, d_traj ? d_traj + (size_t)k * 4 * runs : nullptr, nullptr);
        int live = 0;
        TRY(cudaMemcpyAsync(&live, live_count, sizeof(int), cudaMemcpyDeviceToHost, st));
        TRY(cudaStreamSynchronize(st));
        if (live > 0) {
            // from the second step on, the active set certified at the previous step is tried first
            req.count = live; req.warm_in = req.reuse = warm_valid ? 1 : 0;
            rc = q->solve(req, st);
            if (rc != CARMPC_OK) { cleanup(); return rc; }
            warm_valid = warm != nullptr;
            apply<<<(live + 255) / 256, 256, 0, st>>>(runs, k, live_list, live, nullptr, u0, status, u_prev, d_fail_step, nullptr, gl, inside);
        }
        if (d_u_log)      // the input each run will apply at the next plant step (unchanged for stopped runs)
            TRY(cudaMemcpyAsync(d_u_log + (size_t)k * 2 * runs, u_prev, sizeof(double) * 2 * runs, cudaMemcpyDeviceToDevice, st));
        if (D.dhat_log)   // the estimate the QP of this step used (unchanged for stopped runs)
            TRY(cudaMemcpyAsync(D.dhat_log + (size_t)k * runs, dhat, sizeof(double) * runs, cudaMemcpyDeviceToDevice, st));
    }
    unsigned long long total_dev = 0;
    TRY(cudaMemcpyAsync(&total_dev, q->ws_total_iters, sizeof(total_dev), cudaMemcpyDeviceToHost, st));
    TRY(cudaStreamSynchronize(st));
    total_iters = (int64_t)total_dev;
    TRY(cudaGetLastError());
#undef TRY
    cleanup();
    if (h_total_iters) *h_total_iters = total_iters;
    return CARMPC_OK;
}

// The checks of a monitor's or a goal's row set (nullptr: none); a goal needs d_step and has no d_row.
int check_rows(const carmpc_loop_rows* R, bool goal) {
    if (R == nullptr) return CARMPC_OK;
    const char* use = goal ? "goal" : "monitor";
#define ROWS_REQUIRE(cond, fmt) do { if (!(cond)) { set_error("invalid argument: " fmt, use); return CARMPC_ERR_INVALID; } } while (0)
    ROWS_REQUIRE(R->rows >= 1 && R->rows <= 512, "%s rows must be in [1, 512]");
    ROWS_REQUIRE(R->h_Ab != nullptr, "null %s rows");
    bool finite = true;
    for (int j = 0; j < 5 * R->rows; ++j) finite = finite && isfinite(R->h_Ab[j]);
    ROWS_REQUIRE(finite, "%s rows must be finite");
    ROWS_REQUIRE(!goal || R->d_step != nullptr, "a %s needs d_step");
    ROWS_REQUIRE(!goal || R->d_row == nullptr, "a %s has no d_row");
#undef ROWS_REQUIRE
    return CARMPC_OK;
}

}  // namespace
}  // namespace carmpc

using namespace carmpc;

extern "C" int carmpc_closed_loop(void* qp, int mode, const double* h_A, const double* h_B, const double* h_C,
                                  const double* h_L, const carmpc_disturbance_model* dm, const double* h_xref, double dt,
                                  double l1, int steps, int warm_start, const double* d_x_init, const double* d_xhat_init,
                                  const double* d_dhat_init, const double* d_d_plant, int64_t runs, double* d_final,
                                  double* d_dhat_final, int32_t* d_fail_step, double* d_traj, double* d_u_log,
                                  double* d_dhat_log, const carmpc_loop_noise* noise, const carmpc_loop_rows* monitor,
                                  const carmpc_loop_rows* goal, int64_t* h_total_iters, void* stream) {
    QPHandle* q = check_handle<QPHandle>(qp, kQP);
    CARMPC_REQUIRE(q != nullptr, "not a QP handle");
    CARMPC_REQUIRE(mode >= 0 && mode <= 2, "mode must be 0 (state feedback), 1 (output feedback) or 2 (with a disturbance estimate)");
    CARMPC_REQUIRE(h_A && h_B && h_xref, "null model pointer");
    CARMPC_REQUIRE(mode != 1 || (h_C && h_L), "output feedback needs C and L");
    CARMPC_REQUIRE(mode != 2 || (h_C && dm), "mode 2 needs C and a disturbance model");
    CARMPC_REQUIRE(steps >= 0 && runs >= 0 && runs < (int64_t)1 << 31, "steps / runs");
    CARMPC_REQUIRE(warm_start >= 0 && warm_start <= 2, "warm_start must be 0, 1 or 2");
    CARMPC_REQUIRE(dt > 0 && l1 > 0, "dt, l1");
    bool finite = true;
    if (mode == 1)
        for (int j = 0; j < 12; ++j) finite = finite && isfinite(h_L[j]);
    if (mode == 2) {
        const double* gains[] = {dm->Bd, dm->Cd, dm->L1, dm->L2, dm->Bd_plant, dm->Cd_plant};
        const int counts[] = {4, 3, 12, 3, 4, 3};
        for (int g = 0; g < 6; ++g)
            for (int j = 0; j < counts[g]; ++j) finite = finite && isfinite(gains[g][j]);
    }
    CARMPC_REQUIRE(finite, "observer gains and the disturbance model must be finite");
    if (noise != nullptr) {
        for (int j = 0; j < 16; ++j) finite = finite && isfinite(noise->Lw[j]) && isfinite(noise->Lv[j]);
        CARMPC_REQUIRE(finite, "noise factors Lw, Lv must be finite");
        CARMPC_REQUIRE(noise->first_run >= 0 && noise->first_run <= INT64_MAX - runs, "first_run must be >= 0");
    }
    int rc = check_rows(monitor, false);
    if (rc == CARMPC_OK) rc = check_rows(goal, true);
    if (rc != CARMPC_OK) return rc;
    if (h_total_iters) *h_total_iters = 0;
    if (runs == 0) return CARMPC_OK;
    CARMPC_REQUIRE(d_x_init && d_final && d_fail_step, "null device pointer");
    LoopConst K;
    memset(&K, 0, sizeof(K));
    memcpy(K.A, h_A, sizeof(K.A));
    memcpy(K.B, h_B, sizeof(K.B));
    if (mode != 0) memcpy(K.C, h_C, sizeof(K.C));
    if (mode == 1) memcpy(K.L, h_L, sizeof(K.L));
    LoopDisturbance D = {nullptr, nullptr, nullptr, nullptr};
    if (mode == 2) {
        memcpy(K.L, dm->L1, sizeof(K.L));
        memcpy(K.Bd, dm->Bd, sizeof(K.Bd));
        memcpy(K.Cd, dm->Cd, sizeof(K.Cd));
        memcpy(K.L2, dm->L2, sizeof(K.L2));
        memcpy(K.Bdp, dm->Bd_plant, sizeof(K.Bdp));
        memcpy(K.Cdp, dm->Cd_plant, sizeof(K.Cdp));
        D = {d_dhat_init, d_d_plant, d_dhat_final, d_dhat_log};
    }
    K.dt = dt; K.l1 = l1; K.mode = mode;
    return closed_loop_run(q, K, h_xref, steps, warm_start, d_x_init, d_xhat_init, runs, d_final, d_fail_step, d_traj, d_u_log,
                           D, noise, monitor, goal, h_total_iters, stream);
}
