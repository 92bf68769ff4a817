// Terminal-set membership kernels (K1: H-representation, K2: LQR-rollout form) and their C ABI.
//
// Reference semantics: lib/terminal_set.py:107-113 tests np.all(A @ point <= b) one grid point at a time in a
// Python triple loop.  Here one thread evaluates two samples held in registers, the H-rep rows are broadcast from
// shared memory, the four SoA coordinate arrays are read with 128-bit streaming loads and the result leaves as a
// warp-ballot bitset (1 bit per sample).  Algorithmic HBM traffic: 4 x 8 B read + 1 bit written = 32.125 B / sample.
//
// Arithmetic contract (shared with oracle/carmpc_oracle.c, bit for bit):
//     r = fma(a3, v, fma(a2, psi, fma(a1, y, a0 * x)));   member &= (r <= b);
// in IEEE float64.  Rows are sorted on the host, fewest non-zero coefficients first (for the sets of this model those
// are the axis-aligned bounds on psi, v and y, which reject most samples), so that the whole-warp early exit fires
// soon; the conjunction over rows does not depend on their order.  (A per-pattern specialisation that skipped zero
// coefficients was measured slower than the dense chain: its dispatch cost more issue slots than the FMAs it saved.)
//
// Mode 1 (default) decides almost every sample on the FP32 pipe: it tracks  min_r (b_r - a_r . p)  in float32 (four
// FFMA plus one FMNMX per row) and compares it with a rigorous bound beta(p) on the total rounding error
// of that float32 evaluation; only samples with |min margin| <= beta are re-evaluated in float64 (same bits as mode 0
// by construction).  The FP64 pipe, the co-limiter of mode 0 on B200, stays idle.
#include <math.h>
#include <stdlib.h>

#include <algorithm>
#include <vector>

#include "common.cuh"
#include "shard.cuh"

namespace carmpc {

constexpr int kMaxRows = 512;
constexpr int kThreads = 256;
constexpr int kNS = 4;                                      // samples per thread
constexpr int kChunk = kThreads * kNS;                     // samples per block iteration

// float32 image of one row: negated coefficients and b, so that  margin = fma(-a3, v, ... fma(-a0, x, b))
struct __align__(16) RowF32 {
    float na0, na1, na2, na3;
    float b, pad0, pad1, pad2;
};

// staging geometry of the bulk-async scan: threads per CTA, ring slots per warp, 128-sample tiles per slot
struct Staging {
    int threads = 128, stages = 2, tps = 1;      // measured best of the built geometries on the 10^8 grid (DESIGN.md)
};

// Device staging of the host-buffer entry points: two slots so that the H2D copy of chunk c+1 overlaps the kernel
// and the D2H copy of chunk c.
struct HostStage {
    static constexpr int64_t kChunkSamples = 1 << 23;      // 8 Mi samples: 256 MiB of coordinates per slot
    double* d_coord[2] = {nullptr, nullptr};
    uint32_t* d_bits[2] = {nullptr, nullptr};
    int32_t* d_first[2] = {nullptr, nullptr};
    unsigned long long* d_count = nullptr;
    unsigned long long* d_work = nullptr;                  // [2][2] work counters of the scan kernel, one pair per slot
    cudaStream_t streams[2] = {nullptr, nullptr};
    bool ready = false;
    int64_t cap = 0, first_cap = 0;                        // samples per slot the buffers are sized for
    // Slots are sized to the call (a 60,000-point visualise_set grid takes 2 MB, not the 0.55 GB of two full chunks) and
    // grow on demand up to kChunkSamples; a call that fits one chunk uses one slot.
    int init(bool with_first, int64_t n) {
        if (!ready) {
            for (int i = 0; i < 2; ++i) CARMPC_CUDA(cudaStreamCreateWithFlags(&streams[i], cudaStreamNonBlocking));
            CARMPC_CUDA(cudaMalloc(&d_count, sizeof(unsigned long long)));
            CARMPC_CUDA(cudaMalloc(&d_work, sizeof(unsigned long long) * 4));
            CARMPC_CUDA(cudaMemset(d_work, 0, sizeof(unsigned long long) * 4));
            ready = true;
        }
        const int64_t need = std::min<int64_t>(kChunkSamples, (std::max<int64_t>(n, 1) + 1023) / 1024 * 1024);
        const int slots = n > kChunkSamples ? 2 : 1;
        if (need > cap || (slots == 2 && d_coord[1] == nullptr)) {
            const int64_t sz = std::max(need, cap);
            for (int i = 0; i < 2; ++i) {
                cudaFree(d_coord[i]); cudaFree(d_bits[i]); cudaFree(d_first[i]);
                d_coord[i] = nullptr; d_bits[i] = nullptr; d_first[i] = nullptr;
            }
            cap = 0; first_cap = 0;
            for (int i = 0; i < slots; ++i) {
                CARMPC_CUDA(cudaMalloc(&d_coord[i], sizeof(double) * 4 * sz));
                CARMPC_CUDA(cudaMalloc(&d_bits[i], sizeof(uint32_t) * (sz / 32)));
            }
            cap = sz;
        }
        if (with_first && first_cap < cap) {
            for (int i = 0; i < 2; ++i) { cudaFree(d_first[i]); d_first[i] = nullptr; }
            for (int i = 0; i < 2; ++i)
                if (d_coord[i] != nullptr) CARMPC_CUDA(cudaMalloc(&d_first[i], sizeof(int32_t) * cap));
            first_cap = cap;
        }
        return CARMPC_OK;
    }
    ~HostStage() {
        for (int i = 0; i < 2; ++i) {
            cudaFree(d_coord[i]);
            cudaFree(d_bits[i]);
            cudaFree(d_first[i]);
            if (streams[i]) cudaStreamDestroy(streams[i]);
        }
        cudaFree(d_count);
        cudaFree(d_work);
    }
};

struct Polytope : HandleBase {
    int rows = 0;
    double* d_rows = nullptr;        // rows x 5 (float64), sorted by sparsity pattern
    RowF32* d_rows32 = nullptr;      // rows
    float beta0 = 0.f, beta1 = 0.f;  // |float32 margin - exact margin| <= beta0 + beta1 * max|coordinate|
    HostStage stage;
    std::vector<double> h_rows;      // rows x 5 in device order (host copy, for re-ordering)
    bool tuned = false;              // row order already adapted to a sample set
    Staging staging;                 // geometry of the bulk-async scan (carmpc_scan_staging)
    unsigned long long* d_work = nullptr;   // [2] work counters of the scan kernel (self-resetting)
    double* d_axes = nullptr;        // grid axes of carmpc_membership_grid (4 x 4096 doubles at most)
    double* h_axes = nullptr;        // pinned staging copy
    ~Polytope() override {
        cudaFree(d_rows);
        cudaFree(d_rows32);
        cudaFree(d_axes);
        cudaFreeHost(h_axes);
        cudaFree(d_work);
    }
};

struct Rollout : HandleBase {
    int s = 0, rin = 0, k_steps = 0, input_mode = 0;
    double* d_data = nullptr;        // [Ak 16 | goal 4 | Acon s*4 | bcon s | Ain rin*4 | bin rin]
    RowF32* d_rows32 = nullptr;      // float32 screen: expanded rows a_r A_k^t in absolute coordinates (null: exact kernel only)
    int rows_padded = 0, rows32 = 0;
    float beta0 = 0.f, beta1 = 0.f;
    float in0 = 0.f, in1 = 0.f;      // acceptance band (= beta unless the screen was reduced to the irredundant rows)
    std::vector<double> h_rows64;    // every expanded row as built: [rows][5] = g (4), b' (absolute coordinates)
    std::vector<RowF32> h_rows32;    // host copy (re-ordered by the pilot)
    bool tuned = false;
    Staging staging;
    unsigned long long* d_work = nullptr;
    HostStage stage;
    ~Rollout() override { cudaFree(d_data); cudaFree(d_rows32); cudaFree(d_work); }
};

// spread the 8 bits of a byte to every fourth bit position (bit j -> bit 4 j)
__device__ __forceinline__ uint32_t spread8x4(uint32_t v) {
    v &= 0xffu;
    v = (v | (v << 12)) & 0x000f000fu;
    v = (v | (v << 6)) & 0x03030303u;
    v = (v | (v << 3)) & 0x11111111u;
    return v;
}

struct ScreenConst {         // float32 error-bound constants of the polytope
    float beta0, beta1;      // a sample is surely outside when its smallest margin is below -(beta0 + beta1 |p|_1)
    float in0, in1;          // ... and surely inside when it is above in0 + in1 |p|_1 (= the beta pair, unless the screen only
                             // holds the irredundant rows of the set: then the dropped rows' certificates widen it)
};

constexpr int kExit64 = 4;       // rows between "whole warp already outside" votes, float64 path
constexpr int kRowBlock = 8;     // ... float32 screen (the float32 row image is padded to a multiple of it)

// Largest bound beta(p) = beta0 + beta1 |p|_1 for which the screen may decide.  Every intermediate of a row's float32 chain
// is at most (|b_r| + sum |a_rk| |p_k|) (1 + 2^-21) <= (bmax + l1max |p|_1) (1 + 2^-21), and the constants are built with
// beta0 >= 8 u bmax, beta1 >= 8 u l1max (8 u = 2^-21), so that sum is at most beta(p) 2^21.  At beta(p) <= 1e31 it is below
// 2.2e37 < FLT_MAX / 15: no product or partial sum can overflow to +-inf, which the rounding bound does not cover.
constexpr float kScreenMaxBound = 1e31f;

// float64 decision of the NS samples of this thread: the contract chain, every row, rows in host-sorted order
__device__ __forceinline__ void decide64(const double* __restrict__ s_rows, int rows, const double (&x)[kNS],
                                         const double (&y)[kNS], const double (&p)[kNS], const double (&v)[kNS],
                                         bool (&in)[kNS]) {
    for (int r0 = 0; r0 < rows; r0 += kExit64) {
        bool any = false;
#pragma unroll
        for (int k = 0; k < kNS; ++k) any |= in[k];
        if (!__any_sync(0xffffffffu, any)) break;
        const int r1 = min(r0 + kExit64, rows);
        for (int r = r0; r < r1; ++r) {
            const double* a = s_rows + 5 * r;
            const double a0 = a[0], a1 = a[1], a2 = a[2], a3 = a[3], b = a[4];
#pragma unroll
            for (int k = 0; k < kNS; ++k) in[k] &= (fma(a3, v[k], fma(a2, p[k], fma(a1, y[k], a0 * x[k]))) <= b);
        }
    }
}

// What the float64 decision works on: KIND 0 = the H-rep rows (rows x 5), KIND 1 = the rollout data
// [Ak 16 | goal 4 | Acon s*4 | bcon s | Ain rin*4 | bin rin] (the float32 screen then runs on the expanded rows a_r A_k^t).
struct ExactSpec {
    int len;                 // doubles staged in shared memory
    int rows;                // KIND 0
    int s, rin, k_steps, input_mode;   // KIND 1
};

// float64 decision of the rollout form for the NS samples of this thread: the contract chain of rollout_kernel
// (oracle/carmpc_oracle.c, lib/terminal_set.py:53-59 sampled), step by step
__device__ __forceinline__ void rollout64(const double* __restrict__ s_data, const ExactSpec& es, const double (&x)[kNS],
                                          const double (&y)[kNS], const double (&p)[kNS], const double (&v)[kNS],
                                          bool (&in)[kNS]) {
    const double* Ak = s_data;
    const double* goal = s_data + 16;
    const double* Acon = s_data + 20;
    const double* bcon = Acon + 4 * es.s;
    const double* Ain = bcon + es.s;
    const double* bin = Ain + 4 * es.rin;
    double e0[kNS], e1[kNS], e2[kNS], e3[kNS];
#pragma unroll
    for (int k = 0; k < kNS; ++k) { e0[k] = x[k] - goal[0]; e1[k] = y[k] - goal[1]; e2[k] = p[k] - goal[2]; e3[k] = v[k] - goal[3]; }
    for (int t = 0; t <= es.k_steps; ++t) {
        bool any = false;
#pragma unroll
        for (int k = 0; k < kNS; ++k) any |= in[k];
        if (!__any_sync(0xffffffffu, any)) break;
        for (int r = 0; r < es.s; ++r) {
            const double* a = Acon + 4 * r;
            const double a0 = a[0], a1 = a[1], a2 = a[2], a3 = a[3], b = bcon[r];
#pragma unroll
            for (int k = 0; k < kNS; ++k) in[k] &= (fma(a3, e3[k], fma(a2, e2[k], fma(a1, e1[k], a0 * e0[k]))) <= b);
        }
        if (t == 0 || es.input_mode == 1) {
            for (int r = 0; r < es.rin; ++r) {
                const double* a = Ain + 4 * r;
                const double a0 = a[0], a1 = a[1], a2 = a[2], a3 = a[3], b = bin[r];
#pragma unroll
                for (int k = 0; k < kNS; ++k) in[k] &= (fma(a3, e3[k], fma(a2, e2[k], fma(a1, e1[k], a0 * e0[k]))) <= b);
            }
        }
#pragma unroll
        for (int k = 0; k < kNS; ++k) {
            const double n0 = fma(Ak[3], e3[k], fma(Ak[2], e2[k], fma(Ak[1], e1[k], Ak[0] * e0[k])));
            const double n1 = fma(Ak[7], e3[k], fma(Ak[6], e2[k], fma(Ak[5], e1[k], Ak[4] * e0[k])));
            const double n2 = fma(Ak[11], e3[k], fma(Ak[10], e2[k], fma(Ak[9], e1[k], Ak[8] * e0[k])));
            const double n3 = fma(Ak[15], e3[k], fma(Ak[14], e2[k], fma(Ak[13], e1[k], Ak[12] * e0[k])));
            e0[k] = n0; e1[k] = n1; e2[k] = n2; e3[k] = n3;
        }
    }
}

template <int KIND>
__device__ __forceinline__ void decide_exact(const double* __restrict__ s_rows, const ExactSpec& es, const double (&x)[kNS],
                                             const double (&y)[kNS], const double (&p)[kNS], const double (&v)[kNS],
                                             bool (&in)[kNS]) {
    if (KIND == 0) decide64(s_rows, es.rows, x, y, p, v, in);
    else rollout64(s_rows, es, x, y, p, v, in);
}

// float32 screen: in[k] becomes "surely inside"; returns through amb[k] the samples only the float64 chain can decide
__device__ __forceinline__ void screen32(const RowF32* __restrict__ s_rows32, int rows_padded, const ScreenConst sc,
                                         const float (&xf)[kNS], const float (&yf)[kNS], const float (&pf)[kNS],
                                         const float (&vf)[kNS], bool (&in)[kNS], bool (&amb)[kNS]) {
    float nbeta[kNS], ibeta[kNS], mmin[kNS];
#pragma unroll
    for (int k = 0; k < kNS; ++k) {
        // |x| + |y| + |psi| + |v| >= max |coordinate|, and (unlike fmaxf) it propagates NaN / inf into the bound
        const float psum = (fabsf(xf[k]) + fabsf(yf[k])) + (fabsf(pf[k]) + fabsf(vf[k]));
        nbeta[k] = -fmaf(sc.beta1, psum, sc.beta0);
        ibeta[k] = fmaf(sc.in1, psum, sc.in0);
        mmin[k] = in[k] ? kScreenMaxBound : -INFINITY;       // padding lanes count as "already outside"; for the cap see below
    }
    // samples in pairs: the four fmas of a row run as FFMA2 (same IEEE result per sample as fmaf, half the issue slots)
    f32x2 x2[kNS / 2], y2[kNS / 2], p2[kNS / 2], v2[kNS / 2];
#pragma unroll
    for (int k = 0; k < kNS / 2; ++k) {
        x2[k] = pack2(xf[2 * k], xf[2 * k + 1]); y2[k] = pack2(yf[2 * k], yf[2 * k + 1]);
        p2[k] = pack2(pf[2 * k], pf[2 * k + 1]); v2[k] = pack2(vf[2 * k], vf[2 * k + 1]);
    }
    for (int r0 = 0; r0 < rows_padded; r0 += kRowBlock) {
        bool all_out = true;
#pragma unroll
        for (int k = 0; k < kNS; ++k) all_out &= mmin[k] < nbeta[k];
        if (__all_sync(0xffffffffu, all_out)) break;          // every sample of the warp already surely outside
#pragma unroll
        for (int r = 0; r < kRowBlock; ++r) {
            const RowF32 q = s_rows32[r0 + r];
            const f32x2 a0 = pack2(q.na0, q.na0), a1 = pack2(q.na1, q.na1), a2 = pack2(q.na2, q.na2), a3 = pack2(q.na3, q.na3);
            const f32x2 b = pack2(q.b, q.b);
#pragma unroll
            for (int k = 0; k < kNS / 2; ++k) {
                const f32x2 m2 = ffma2(a3, v2[k], ffma2(a2, p2[k], ffma2(a1, y2[k], ffma2(a0, x2[k], b))));
                float m_lo, m_hi;
                unpack2(m2, m_lo, m_hi);
                mmin[2 * k] = fminf(mmin[2 * k], m_lo);       // a NaN margin is ignored here; NaN inputs are caught by the bound
                mmin[2 * k + 1] = fminf(mmin[2 * k + 1], m_hi);
            }
        }
    }
#pragma unroll
    for (int k = 0; k < kNS; ++k) {
        // No decision where the bound exceeds kScreenMaxBound or is NaN: the float32 chain may have overflowed (its margin
        // can be a wrong +-inf; the early exit above may act on it, which only skips rows), the coordinates are not finite,
        // or the beta pair is infinite because the rows have no faithful float32 image.  The float64 chain decides those.
        // "Surely inside" needs mmin > ibeta >= bound, and mmin never exceeds its start value kScreenMaxBound, so only
        // "surely outside" needs the explicit test (one compare per sample instead of two).
        const bool sure_in = mmin[k] > ibeta[k], sure_out = mmin[k] < nbeta[k] && nbeta[k] >= -kScreenMaxBound;
        amb[k] = in[k] && !sure_in && !sure_out;
        in[k] = in[k] && sure_in;
    }
}

// Where the bitset words of a scan go.  One destination for a plain call; for a scan that is one shard of a sample set
// partitioned over the GPUs of a box, one destination per rank (the rank's own full bitset and, through NVLink peer
// mappings, every other rank's), each already pointing at the first word of this shard - the scan kernel itself
// performs the all-gather (SURVEY 8e), no separate collective.
// Layout: the k-th 1024-sample group of the scanned arrays is group k * stride of the destination bitsets (stride 1:
// a contiguous shard; stride = number of ranks: the groups of the sample set are dealt round-robin to the ranks, which
// balances the load when the cost of a sample depends on where it lies).
constexpr int kMaxPeers = 8;
struct BitSink {
    uint32_t* dst[kMaxPeers];
    int n;
    int64_t stride;
    // double-buffered destinations (peer windows): the buffer of this launch is slot (*step + 1) & 1, slot_words apart.
    // The step lives in device memory (advanced by the exchange kernel), so the launch arguments of a collective step
    // never change and the step can be captured in a CUDA graph.  nullptr: single buffer.
    const unsigned long long* step;
    int64_t slot_words;
};

__device__ __forceinline__ int64_t sink_slot_offset(const BitSink& sink) {
    return sink.step != nullptr ? (int64_t)((*sink.step + 1ull) & 1ull) * sink.slot_words : 0;
}

static BitSink single_sink(uint32_t* bits) {
    BitSink s{};
    s.dst[0] = bits;
    s.n = 1;
    s.stride = 1;
    s.step = nullptr;
    s.slot_words = 0;
    return s;
}

// the sink of the samples that follow `groups` whole local groups
static BitSink offset_sink(const BitSink& in, int64_t groups) {
    BitSink s = in;
    for (int d = 0; d < s.n; ++d) s.dst[d] += groups * in.stride * 32;
    return s;
}

// destination word of local word wl (32 words per group)
__device__ __forceinline__ int64_t sink_word(const BitSink& sink, int64_t wl) {
    return sink.stride == 1 ? wl : ((wl >> 5) * sink.stride << 5) + (wl & 31);
}

// The 128 decisions of a warp tile (lane t holds samples 4t .. 4t+3) as four words: returns to EVERY lane the word
// (lane & 3) of the tile, and the number of members through `members`.
__device__ __forceinline__ uint32_t tile_word(const bool (&in)[kNS], int& members) {
    uint32_t bal[kNS];
#pragma unroll
    for (int k = 0; k < kNS; ++k) {
        bal[k] = __ballot_sync(0xffffffffu, in[k]);
        members += __popc(bal[k]);
    }
    const int q = threadIdx.x & 3;
    uint32_t word = 0;
#pragma unroll
    for (int k = 0; k < kNS; ++k) word |= spread8x4(bal[k] >> (8 * q)) << k;
    return word;
}

// write the 128 decisions of a warp (lane t holds samples 4t .. 4t+3 of the warp's chunk) as four words
__device__ __forceinline__ int store_bits(const BitSink& sink, int64_t warp_base, int64_t n, const bool (&in)[kNS]) {
    int members = 0;
    const uint32_t word = tile_word(in, members);
    const int lane = threadIdx.x & 31;
    if (lane < 4) {
        const int64_t first = warp_base + 32 * lane;
        if (first < n) {
            const int64_t wg = sink_word(sink, first >> 5) + sink_slot_offset(sink);
#pragma unroll
            for (int d = 0; d < kMaxPeers; ++d)
                if (d < sink.n) sink.dst[d][wg] = word;
        }
    }
    return members;
}

template <int THREADS = kThreads>
__device__ __forceinline__ void block_count(int warp_members, unsigned long long* __restrict__ count) {
    __shared__ int s_partial[THREADS / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0) s_partial[warp] = warp_members;
    __syncthreads();
    if (threadIdx.x == 0 && count != nullptr) {
        int total = 0;
#pragma unroll
        for (int w = 0; w < THREADS / 32; ++w) total += s_partial[w];
        if (total) atomicAdd(count, (unsigned long long)total);
    }
}

__device__ __forceinline__ void stage_rows(const double* __restrict__ g_rows, const RowF32* __restrict__ g_rows32,
                                           int exact_len, int rows_padded, double* s_rows, RowF32* s_rows32) {
    for (int i = threadIdx.x; i < exact_len; i += blockDim.x) s_rows[i] = g_rows[i];
    for (int i = threadIdx.x; i < rows_padded; i += blockDim.x) s_rows32[i] = g_rows32[i];
    __syncthreads();
}

// four consecutive samples of one coordinate array (two 128-bit streaming loads when aligned and in range)
template <bool VEC>
__device__ __forceinline__ void load4(const double* __restrict__ g, int64_t i0, int64_t n, double (&out)[kNS]) {
    if (VEC && i0 + 3 < n) {
        const double2 a = ld_stream_f64x2(g + i0), b = ld_stream_f64x2(g + i0 + 2);
        out[0] = a.x; out[1] = a.y; out[2] = b.x; out[3] = b.y;
    } else {
#pragma unroll
        for (int k = 0; k < kNS; ++k) out[k] = i0 + k < n ? ld_stream_f64(g + i0 + k) : 0.0;
    }
}

template <int MODE, bool VEC, int KIND>
__global__ void __launch_bounds__(kThreads)
membership_kernel(const double* __restrict__ g_rows, const RowF32* __restrict__ g_rows32, const ExactSpec es, int rows_padded,
                  const ScreenConst sc, const double* __restrict__ gx, const double* __restrict__ gy,
                  const double* __restrict__ gp, const double* __restrict__ gv, int64_t n,
                  const BitSink sink, unsigned long long* __restrict__ count) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    double* s_rows = reinterpret_cast<double*>(smem_raw);
    RowF32* s_rows32 = reinterpret_cast<RowF32*>(s_rows + ((es.len + 1) & ~1));
    stage_rows(g_rows, g_rows32, es.len, rows_padded, s_rows, s_rows32);

    int members = 0;
    const int64_t n_chunks = (n + kChunk - 1) / kChunk;
    for (int64_t chunk = blockIdx.x; chunk < n_chunks; chunk += gridDim.x) {
        const int64_t i0 = chunk * kChunk + kNS * (int64_t)threadIdx.x;
        bool in[kNS];
#pragma unroll
        for (int k = 0; k < kNS; ++k) in[k] = i0 + k < n;
        if (MODE == 0) {
            double x[kNS], y[kNS], p[kNS], v[kNS];
            load4<VEC>(gx, i0, n, x); load4<VEC>(gy, i0, n, y); load4<VEC>(gp, i0, n, p); load4<VEC>(gv, i0, n, v);
            decide_exact<KIND>(s_rows, es, x, y, p, v, in);
        } else {
            float xf[kNS], yf[kNS], pf[kNS], vf[kNS];
            {
                double x[kNS], y[kNS], p[kNS], v[kNS];
                load4<VEC>(gx, i0, n, x); load4<VEC>(gy, i0, n, y); load4<VEC>(gp, i0, n, p); load4<VEC>(gv, i0, n, v);
#pragma unroll
                for (int k = 0; k < kNS; ++k) { xf[k] = (float)x[k]; yf[k] = (float)y[k]; pf[k] = (float)p[k]; vf[k] = (float)v[k]; }
            }
            bool amb[kNS];
            screen32(s_rows32, rows_padded, sc, xf, yf, pf, vf, in, amb);
            bool any_amb = false;
#pragma unroll
            for (int k = 0; k < kNS; ++k) any_amb |= amb[k];
            if (__any_sync(0xffffffffu, any_amb)) {
                // rare (|margin| <= beta, ~1e-5 relative, or a non-finite coordinate): the float64 coordinates are
                // read again (L2) and the float64 chain decides, exactly as in mode 0
                double x[kNS], y[kNS], p[kNS], v[kNS];
                load4<VEC>(gx, i0, n, x); load4<VEC>(gy, i0, n, y); load4<VEC>(gp, i0, n, p); load4<VEC>(gv, i0, n, v);
                decide_exact<KIND>(s_rows, es, x, y, p, v, amb);
#pragma unroll
                for (int k = 0; k < kNS; ++k) in[k] |= amb[k];
            }
        }
        const int64_t warp_base = chunk * kChunk + 32 * kNS * (int64_t)(threadIdx.x >> 5);
        members += store_bits(sink, warp_base, n, in);
    }
    block_count(members, count);
}

// ---- bulk-async (TMA) staged variant ---------------------------------------------------------------------------------
// The scan is HBM-bound, and with plain loads the bytes in flight are limited by the registers that receive them
// (8 x 128-bit loads per thread) times the occupancy.  Here every warp runs its own STAGES-deep shared-memory ring: lane 0
// streams the warp's next stage (4 arrays x TPS tiles x 128 samples x 8 B) with cp.async.bulk, completion is tracked by
// one mbarrier per stage (expect_tx / complete_tx), the warp waits on the stage, pulls its samples into registers,
// __syncwarp()s, and lane 0 immediately refills the stage.  Warps never wait for each other (the early exits make
// their tiles very unequal), and the bytes in flight do not depend on register allocation.
//
// Work unit of a warp: a GROUP of 8 consecutive tiles = 1024 samples = 32 bitset words, handed out round-robin over
// all warps of the grid.  The 32 words of a group are collected one per lane and leave as ONE 128-byte store per
// destination (the local bitset and, for a sharded scan, every peer's copy over NVLink).
constexpr int kTile = 32 * kNS;                 // samples per warp tile
constexpr int kGroupTiles = 8;                  // tiles per group
constexpr int kGroup = kTile * kGroupTiles;     // samples per group (1024)

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_load(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(dst_smem)), "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    uint32_t done = 0;
    int spins = 0;
    while (!done) {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(done) : "r"(smem_u32(bar)), "r"(parity) : "memory");
        if (!done && ++spins > (1 << 24)) __trap();          // a lost transaction must fail loudly, not hang the GPU
    }
}

// THREADS per CTA, STAGES ring slots per warp, TPS tiles (of 128 samples) per slot
template <int MODE, int KIND, int THREADS, int STAGES, int TPS>
__global__ void __launch_bounds__(THREADS)
membership_tma_kernel(const double* __restrict__ g_rows, const RowF32* __restrict__ g_rows32, const ExactSpec es, int rows_padded,
                      const ScreenConst sc, const double* __restrict__ gx, const double* __restrict__ gy,
                      const double* __restrict__ gp, const double* __restrict__ gv, int64_t n_groups,
                      const BitSink sink, unsigned long long* __restrict__ count, unsigned long long* __restrict__ work) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    constexpr int kWarps = THREADS / 32;
    constexpr int kSlot = TPS * kTile;                    // samples per ring slot and array
    constexpr int kSlotsPerGroup = kGroupTiles / TPS;
    static_assert(kGroupTiles % TPS == 0, "a group is a whole number of ring slots");
    double* s_stage = reinterpret_cast<double*>(smem_raw);                       // [kWarps][STAGES][4][kSlot]
    uint64_t* s_bar = reinterpret_cast<uint64_t*>(s_stage + (size_t)kWarps * STAGES * 4 * kSlot);   // [kWarps][STAGES]
    double* s_rows = reinterpret_cast<double*>(s_bar + kWarps * STAGES);
    RowF32* s_rows32 = reinterpret_cast<RowF32*>(s_rows + ((es.len + 1) & ~1));
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const double* src[4] = {gx, gy, gp, gv};
    constexpr uint32_t kArrayBytes = kSlot * sizeof(double);
    double* w_stage = s_stage + (size_t)warp * STAGES * 4 * kSlot;
    uint64_t* w_bar = s_bar + warp * STAGES;

    if (lane == 0) {
        for (int s = 0; s < STAGES; ++s) mbar_init(w_bar + s, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    stage_rows(g_rows, g_rows32, es.len, rows_padded, s_rows, s_rows32);        // ends with __syncthreads()

    // Groups are handed out dynamically (one atomic per 1024 samples): their cost varies a lot (a warp leaves a tile as soon
    // as every sample is rejected) and, on tensor grids, periodically in the sample index, so a static round-robin leaves
    // some warps with systematically more work and the kernel with a long tail.
    // Producer (lane 0): group pg, next slot ps of it, running slot count pj; it is never more than one group ahead of
    // the consumer (STAGES <= slots per group), so the consumer's next group is always the producer's current one.
    static_assert(STAGES <= kSlotsPerGroup, "the producer may be at most one group ahead");
    int64_t pg = 0;
    int ps = 0, pj = 0;
    auto advance = [&]() {                                                       // lane 0: issue the next slot of the sequence
        if (pg >= n_groups) return;
        const int64_t sample = pg * kGroup + (int64_t)ps * kSlot;
        const int stage = pj % STAGES;
        mbar_expect_tx(w_bar + stage, 4 * kArrayBytes);
#pragma unroll
        for (int a = 0; a < 4; ++a)
            bulk_load(w_stage + ((size_t)stage * 4 + a) * kSlot, src[a] + sample, kArrayBytes, w_bar + stage);
        ++pj;
        if (++ps == kSlotsPerGroup) { ps = 0; pg = (int64_t)atomicAdd(work, 1ull); }
    };
    if (lane == 0) pg = (int64_t)atomicAdd(work, 1ull);
    int64_t group = __shfl_sync(0xffffffffu, pg, 0);
    if (lane == 0)
        for (int s = 0; s < STAGES; ++s) advance();

    int members = 0;
    int j = 0;
    const int64_t slot_off = sink_slot_offset(sink);
    while (group < n_groups) {
        uint32_t acc = 0;                                  // lane l collects word l of the group's 32
#pragma unroll 1
        for (int sg = 0; sg < kSlotsPerGroup; ++sg, ++j) {
            const int stage = j % STAGES;
            mbar_wait(w_bar + stage, (uint32_t)(j / STAGES) & 1u);
#pragma unroll
            for (int t = 0; t < TPS; ++t) {
                const double* st = w_stage + (size_t)stage * 4 * kSlot + t * kTile + kNS * lane;
                double x[kNS], y[kNS], p[kNS], v[kNS];
#pragma unroll
                for (int k = 0; k < kNS; k += 2) {
                    const double2 X = *reinterpret_cast<const double2*>(st + k);
                    const double2 Y = *reinterpret_cast<const double2*>(st + kSlot + k);
                    const double2 P = *reinterpret_cast<const double2*>(st + 2 * kSlot + k);
                    const double2 V = *reinterpret_cast<const double2*>(st + 3 * kSlot + k);
                    x[k] = X.x; x[k + 1] = X.y; y[k] = Y.x; y[k + 1] = Y.y;
                    p[k] = P.x; p[k + 1] = P.y; v[k] = V.x; v[k + 1] = V.y;
                }
                float xf[kNS], yf[kNS], pf[kNS], vf[kNS];
                if (MODE == 1) {
#pragma unroll
                    for (int k = 0; k < kNS; ++k) { xf[k] = (float)x[k]; yf[k] = (float)y[k]; pf[k] = (float)p[k]; vf[k] = (float)v[k]; }
                }
                if (t == TPS - 1) {
                    __syncwarp();                          // every lane has the slot's last samples in registers: slot is free
                    if (lane == 0) advance();
                }
                bool in[kNS];
#pragma unroll
                for (int k = 0; k < kNS; ++k) in[k] = true;
                if (MODE == 0) {
                    decide_exact<KIND>(s_rows, es, x, y, p, v, in);
                } else {
                    bool amb[kNS];
                    screen32(s_rows32, rows_padded, sc, xf, yf, pf, vf, in, amb);
                    bool any_amb = false;
#pragma unroll
                    for (int k = 0; k < kNS; ++k) any_amb |= amb[k];
                    if (__any_sync(0xffffffffu, any_amb)) {
                        // rare: re-read the float64 coordinates (L2) and let the float64 chain decide, as in mode 0
                        const int64_t i0 = group * kGroup + (int64_t)(sg * TPS + t) * kTile + kNS * (int64_t)lane;
                        double x2[kNS], y2[kNS], p2[kNS], v2[kNS];
                        load4<true>(gx, i0, n_groups * kGroup, x2); load4<true>(gy, i0, n_groups * kGroup, y2);
                        load4<true>(gp, i0, n_groups * kGroup, p2); load4<true>(gv, i0, n_groups * kGroup, v2);
                        decide_exact<KIND>(s_rows, es, x2, y2, p2, v2, amb);
#pragma unroll
                        for (int k = 0; k < kNS; ++k) in[k] |= amb[k];
                    }
                }
                const uint32_t word = tile_word(in, members);
                if ((lane >> 2) == sg * TPS + t) acc = word;
            }
        }
        const int64_t w0 = slot_off + group * sink.stride * (kGroup / 32) + lane;
#pragma unroll
        for (int d = 0; d < kMaxPeers; ++d)
            if (d < sink.n) sink.dst[d][w0] = acc;
        group = __shfl_sync(0xffffffffu, pg, 0);           // all slots of the finished group were issued: pg is its successor
    }
    block_count<THREADS>(members, count);                  // ends after a __syncthreads(): every warp of the CTA is done
    // the last CTA to finish re-arms the work counter for the next launch
    if (tid == 0) {
        __threadfence();
        if (atomicAdd(work + 1, 1ull) == (unsigned long long)gridDim.x - 1ull) {
            work[0] = 0ull;
            work[1] = 0ull;
            __threadfence();
        }
    }
}

struct GridDesc {
    int32_t dims[4];
    int32_t state_of_axis[4];
    int32_t offset[4];      // start of each axis in the concatenated axes array
};

// implicit tensor grid: coordinates come from four short axes staged in shared memory, no HBM reads at all
__global__ void __launch_bounds__(kThreads, 4)        // 4 CTAs per SM: the launch below sizes the grid for that
membership_grid_kernel(const double* __restrict__ g_rows, const RowF32* __restrict__ g_rows32, int rows, int rows_padded,
                       const ScreenConst sc, const double* __restrict__ g_axes, GridDesc gd, int64_t n,
                       uint32_t* __restrict__ bits, unsigned long long* __restrict__ count) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    double* s_rows = reinterpret_cast<double*>(smem_raw);
    RowF32* s_rows32 = reinterpret_cast<RowF32*>(s_rows + ((rows * 5 + 1) & ~1));
    double* s_axes = reinterpret_cast<double*>(s_rows32 + rows_padded);
    const int axes_len = gd.offset[3] + gd.dims[3];
    float* s_axes32 = reinterpret_cast<float*>(s_axes + axes_len);          // float32 images for the screen (converted once)
    for (int i = threadIdx.x; i < axes_len; i += blockDim.x) { const double a = g_axes[i]; s_axes[i] = a; s_axes32[i] = (float)a; }
    stage_rows(g_rows, g_rows32, rows * 5, rows_padded, s_rows, s_rows32);

    int members = 0;
    const int64_t n_chunks = (n + kChunk - 1) / kChunk;
    for (int64_t chunk = blockIdx.x; chunk < n_chunks; chunk += gridDim.x) {
        const int64_t i0 = chunk * kChunk + kNS * (int64_t)threadIdx.x;
        bool in[kNS];
        // multi-index of the thread's first sample: one decomposition per chunk (32-bit divisions when the grid allows),
        // the following kNS - 1 samples by incrementing with carry
        uint32_t idx0[4];
        {
            const uint64_t first = i0 < n ? (uint64_t)i0 : 0;
            if (n <= 0xffffffffll) {
                uint32_t rem = (uint32_t)first;
#pragma unroll
                for (int ax = 3; ax >= 1; --ax) {
                    const uint32_t d = (uint32_t)gd.dims[ax], qd = rem / d;
                    idx0[ax] = rem - qd * d;
                    rem = qd;
                }
                idx0[0] = rem;
            } else {
                uint64_t rem = first;
#pragma unroll
                for (int ax = 3; ax >= 1; --ax) {
                    const uint32_t d = (uint32_t)gd.dims[ax];
                    const uint64_t qd = rem / d;
                    idx0[ax] = (uint32_t)(rem - qd * d);
                    rem = qd;
                }
                idx0[0] = (uint32_t)rem;
            }
        }
        auto advance = [&](uint32_t (&idx)[4]) {
            if (++idx[3] == (uint32_t)gd.dims[3]) {
                idx[3] = 0;
                if (++idx[2] == (uint32_t)gd.dims[2]) {
                    idx[2] = 0;
                    if (++idx[1] == (uint32_t)gd.dims[1]) { idx[1] = 0; ++idx[0]; }       // past the end: clamped below, masked by in[]
                }
            }
        };
        float cf[4][kNS];
        {
            uint32_t idx[4] = {idx0[0], idx0[1], idx0[2], idx0[3]};
#pragma unroll
            for (int k = 0; k < kNS; ++k) {
                in[k] = i0 + k < n;
#pragma unroll
                for (int ax = 0; ax < 4; ++ax) {
                    const float val = s_axes32[gd.offset[ax] + min(idx[ax], (uint32_t)gd.dims[ax] - 1u)];
                    // state_of_axis is a permutation of 0..3
#pragma unroll
                    for (int st = 0; st < 4; ++st)
                        if (gd.state_of_axis[ax] == st) cf[st][k] = val;
                }
                advance(idx);
            }
        }
        bool amb[kNS];
        screen32(s_rows32, rows_padded, sc, cf[0], cf[1], cf[2], cf[3], in, amb);
        bool any_amb = false;
#pragma unroll
        for (int k = 0; k < kNS; ++k) any_amb |= amb[k];
        if (__any_sync(0xffffffffu, any_amb)) {
            // the float64 coordinates are only needed for the samples the screen could not decide
            double c[4][kNS];
            uint32_t idx[4] = {idx0[0], idx0[1], idx0[2], idx0[3]};
#pragma unroll
            for (int k = 0; k < kNS; ++k) {
#pragma unroll
                for (int ax = 0; ax < 4; ++ax) {
                    const double val = s_axes[gd.offset[ax] + min(idx[ax], (uint32_t)gd.dims[ax] - 1u)];
#pragma unroll
                    for (int st = 0; st < 4; ++st)
                        if (gd.state_of_axis[ax] == st) c[st][k] = val;
                }
                advance(idx);
            }
            decide64(s_rows, rows, c[0], c[1], c[2], c[3], amb);
#pragma unroll
            for (int k = 0; k < kNS; ++k) in[k] |= amb[k];
        }
        const int64_t warp_base = chunk * kChunk + 32 * kNS * (int64_t)(threadIdx.x >> 5);
        BitSink sink;
        sink.dst[0] = bits;
        sink.n = 1;
        sink.stride = 1;
        sink.step = nullptr;
        sink.slot_words = 0;
        members += store_bits(sink, warp_base, n, in);
    }
    block_count(members, count);
}

// ---- K2: rollout form --------------------------------------------------------------------------------------------------
// one sample per thread; e (4 registers) is propagated k_steps times by A_k, rows are broadcast from shared memory.
__global__ void __launch_bounds__(kThreads)
rollout_kernel(const double* __restrict__ g_data, int s, int rin, int k_steps, int input_mode,
               const double* __restrict__ gx, const double* __restrict__ gy, const double* __restrict__ gp,
               const double* __restrict__ gv, int64_t n, const BitSink sink,
               int32_t* __restrict__ first_violation, unsigned long long* __restrict__ count) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    double* s_data = reinterpret_cast<double*>(smem_raw);
    const int total = 20 + 5 * s + 5 * rin;
    for (int i = threadIdx.x; i < total; i += blockDim.x) s_data[i] = g_data[i];
    __syncthreads();
    const double* Ak = s_data;
    const double* goal = s_data + 16;
    const double* Acon = s_data + 20;
    const double* bcon = Acon + 4 * s;
    const double* Ain = bcon + s;
    const double* bin = Ain + 4 * rin;

    int members = 0;
    const int64_t n_chunks = (n + kThreads - 1) / kThreads;
    for (int64_t chunk = blockIdx.x; chunk < n_chunks; chunk += gridDim.x) {
        const int64_t i = chunk * kThreads + threadIdx.x;
        const bool valid = i < n;
        const int64_t j = valid ? i : 0;
        double e0 = ld_stream_f64(gx + j) - goal[0];
        double e1 = ld_stream_f64(gy + j) - goal[1];
        double e2 = ld_stream_f64(gp + j) - goal[2];
        double e3 = ld_stream_f64(gv + j) - goal[3];
        bool in = valid;
        int first = -1;
        for (int t = 0; t <= k_steps; ++t) {
            if (!__any_sync(0xffffffffu, in)) break;
            bool ok = true;
            for (int r = 0; r < s; ++r) {
                const double* a = Acon + 4 * r;
                const double rr = fma(a[3], e3, fma(a[2], e2, fma(a[1], e1, a[0] * e0)));
                ok &= (rr <= bcon[r]);
            }
            if (t == 0 || input_mode == 1) {
                for (int r = 0; r < rin; ++r) {
                    const double* a = Ain + 4 * r;
                    const double rr = fma(a[3], e3, fma(a[2], e2, fma(a[1], e1, a[0] * e0)));
                    ok &= (rr <= bin[r]);
                }
            }
            if (in && !ok) first = t;
            in &= ok;
            const double n0 = fma(Ak[3], e3, fma(Ak[2], e2, fma(Ak[1], e1, Ak[0] * e0)));
            const double n1 = fma(Ak[7], e3, fma(Ak[6], e2, fma(Ak[5], e1, Ak[4] * e0)));
            const double n2 = fma(Ak[11], e3, fma(Ak[10], e2, fma(Ak[9], e1, Ak[8] * e0)));
            const double n3 = fma(Ak[15], e3, fma(Ak[14], e2, fma(Ak[13], e1, Ak[12] * e0)));
            e0 = n0; e1 = n1; e2 = n2; e3 = n3;
        }
        const uint32_t word = __ballot_sync(0xffffffffu, in);
        if ((threadIdx.x & 31) == 0 && i < n) {
            const int64_t wg = sink_word(sink, i >> 5) + sink_slot_offset(sink);
#pragma unroll
            for (int d = 0; d < kMaxPeers; ++d)
                if (d < sink.n) sink.dst[d][wg] = word;
        }
        if (first_violation != nullptr && valid) first_violation[i] = first;
        if ((threadIdx.x & 31) == 0) members += __popc(word);
    }
    // members is only non-zero on lane 0 of each warp here
    __shared__ int s_partial[kThreads / 32];
    if ((threadIdx.x & 31) == 0) s_partial[threadIdx.x >> 5] = members;
    __syncthreads();
    if (threadIdx.x == 0 && count != nullptr) {
        int total_members = 0;
        for (int w = 0; w < kThreads / 32; ++w) total_members += s_partial[w];
        if (total_members) atomicAdd(count, (unsigned long long)total_members);
    }
}

// ---- host side -----------------------------------------------------------------------------------------------------------
static int pad_rows(int rows) { return (rows + 7) & ~7; }
static size_t membership_smem(int rows) { return sizeof(double) * ((rows * 5 + 1) & ~1) + sizeof(RowF32) * pad_rows(rows); }   // grid kernel

static int grid_blocks(int64_t n_chunks, int per_sm) {
    const int64_t cap = (int64_t)sm_count() * per_sm;
    return (int)(n_chunks < cap ? (n_chunks > 0 ? n_chunks : 1) : cap);
}

static ScreenConst screen_const(const Polytope* P) {
    ScreenConst sc;
    sc.beta0 = P->beta0;
    sc.beta1 = P->beta1;
    sc.in0 = P->beta0;
    sc.in1 = P->beta1;
    return sc;
}

static size_t scan_smem(int exact_len, int rows_padded) {
    return sizeof(double) * ((exact_len + 1) & ~1) + sizeof(RowF32) * rows_padded;
}
static size_t scan_tma_smem(int exact_len, int rows_padded, const Staging& g) {
    return sizeof(double) * (g.threads / 32) * g.stages * 4 * g.tps * kTile + sizeof(uint64_t) * (g.threads / 32) * g.stages +
           scan_smem(exact_len, rows_padded) + 16;
}
static bool staging_supported(const Staging& g) {
    static const int ok[][3] = {{256, 3, 1}, {128, 3, 1}, {128, 4, 1}, {128, 2, 2}, {128, 3, 2}, {256, 2, 1}, {128, 2, 1}, {256, 2, 2}};
    for (const auto& v : ok)
        if (v[0] == g.threads && v[1] == g.stages && v[2] == g.tps) return true;
    return false;
}

template <int KIND, int THREADS, int STAGES, int TPS>
static int launch_tma(const double* d_exact, const RowF32* d_rows32, const ExactSpec& es, int rows_padded, const ScreenConst& sc,
                      const double* x, const double* y, const double* p, const double* v, int64_t n_groups,
                      const BitSink& sink, unsigned long long* count, unsigned long long* work, size_t smem, cudaStream_t st) {
    auto kernel = membership_tma_kernel<1, KIND, THREADS, STAGES, TPS>;
    // the function attribute is per device and the occupancy depends on smem only through the row count, which rarely
    // changes between calls: both are cached per device
    static int per_sm_cached[64];
    static size_t smem_cached[64];
    int dev = 0;
    CARMPC_CUDA(cudaGetDevice(&dev));
    dev &= 63;
    if (per_sm_cached[dev] <= 0 || smem_cached[dev] != smem) {
        CARMPC_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        int per_sm = 0;
        CARMPC_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, THREADS, smem));
        per_sm_cached[dev] = per_sm > 0 ? per_sm : 1;
        smem_cached[dev] = smem;
    }
    const int64_t n_units = (n_groups + THREADS / 32 - 1) / (THREADS / 32);
    kernel<<<grid_blocks(n_units, per_sm_cached[dev]), THREADS, smem, st>>>(d_exact, d_rows32, es, rows_padded, sc, x, y, p, v,
                                                                      n_groups, sink, count, work);
    CARMPC_CUDA(cudaGetLastError());
    return CARMPC_OK;
}

// Streaming scan shared by the H-rep membership (KIND 0) and the screened rollout form (KIND 1).
template <int KIND>
static int launch_scan(const double* d_exact, const RowF32* d_rows32, const ExactSpec es, int rows_padded,
                       const ScreenConst sc, const double* x, const double* y, const double* p, const double* v,
                       int64_t n, BitSink sink, unsigned long long* count, unsigned long long* work, int mode, const Staging& geo,
                       cudaStream_t st) {
    if (n == 0) return CARMPC_OK;
    const bool vec = ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(y) |
                       reinterpret_cast<uintptr_t>(p) | reinterpret_cast<uintptr_t>(v)) & 15) == 0;
    // Bulk-async staged kernel for the whole 1024-sample groups of 16-byte aligned arrays; whatever is left (a ragged
    // tail of fewer than 1024 samples, or unaligned arrays) goes through the plain-load kernel below.
    // (mode 0 is FP64-pipe bound and prefers the higher occupancy of the plain kernel: measured 0.72 vs 0.82 ms)
    if (vec && mode == 1 && n >= 64 * (int64_t)kChunk) {
        const int64_t n_groups = n / kGroup;
        const size_t smem = scan_tma_smem(es.len, rows_padded, geo);
        int rc = CARMPC_ERR_UNSUPPORTED;
#define TMA_CASE(T, S, P)                                                                                              \
        if (geo.threads == T && geo.stages == S && geo.tps == P)                                                           \
            rc = launch_tma<KIND, T, S, P>(d_exact, d_rows32, es, rows_padded, sc, x, y, p, v, n_groups, sink, count, work, smem, st)
        TMA_CASE(256, 3, 1); TMA_CASE(128, 3, 1); TMA_CASE(128, 4, 1); TMA_CASE(128, 2, 2);
        TMA_CASE(128, 3, 2); TMA_CASE(256, 2, 1); TMA_CASE(128, 2, 1); TMA_CASE(256, 2, 2);
#undef TMA_CASE
        if (rc == CARMPC_ERR_UNSUPPORTED) set_error("membership scan: staging geometry %d/%d/%d is not built", geo.threads, geo.stages, geo.tps);
        if (rc != CARMPC_OK) return rc;
        const int64_t done = n_groups * kGroup;
        if (done == n) return CARMPC_OK;
        x += done; y += done; p += done; v += done; n -= done;
        sink = offset_sink(sink, n_groups);
    }
    const size_t smem = scan_smem(es.len, rows_padded);
    const int64_t n_chunks = (n + kChunk - 1) / kChunk;
    // persistent grid: exactly the number of CTAs that are resident at once (a multiple of the SM count)
#define LAUNCH(M, V)                                                                                              \
    do {                                                                                                          \
        int per_sm = 0;                                                                                           \
        CARMPC_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, membership_kernel<M, V, KIND>, kThreads, smem)); \
        const int blocks = grid_blocks(n_chunks, per_sm > 0 ? per_sm : 1);                                        \
        membership_kernel<M, V, KIND><<<blocks, kThreads, smem, st>>>(d_exact, d_rows32, es, rows_padded, sc, x, y, p, v, \
                                                                      n, sink, count);                            \
    } while (0)
    if (mode == 0) {
        if (vec) LAUNCH(0, true); else LAUNCH(0, false);
    } else {
        if (vec) LAUNCH(1, true); else LAUNCH(1, false);
    }
#undef LAUNCH
    CARMPC_CUDA(cudaGetLastError());
    return CARMPC_OK;
}

static int launch_membership(Polytope* P, const double* x, const double* y, const double* p, const double* v,
                             int64_t n, const BitSink& sink, unsigned long long* count, unsigned long long* work, int mode,
                             cudaStream_t st) {
    ExactSpec es{};
    es.len = P->rows * 5;
    es.rows = P->rows;
    return launch_scan<0>(P->d_rows, P->d_rows32, es, pad_rows(P->rows), screen_const(P), x, y, p, v, n, sink, count, work, mode,
                          P->staging, st);
}

static int launch_rollout(Rollout* R, const double* x, const double* y, const double* p, const double* v, int64_t n,
                          const BitSink& sink, int32_t* first, unsigned long long* count, unsigned long long* work, cudaStream_t st) {
    if (n == 0) return CARMPC_OK;
    if (first == nullptr && R->d_rows32 != nullptr) {
        // float32 screen over the expanded rows a_r A_k^t, float64 step-by-step rollout for the samples it cannot decide
        ExactSpec es{};
        es.len = 20 + 5 * R->s + 5 * R->rin;
        es.s = R->s; es.rin = R->rin; es.k_steps = R->k_steps; es.input_mode = R->input_mode;
        ScreenConst sc;
        sc.beta0 = R->beta0; sc.beta1 = R->beta1; sc.in0 = R->in0; sc.in1 = R->in1;
        return launch_scan<1>(R->d_data, R->d_rows32, es, R->rows_padded, sc, x, y, p, v, n, sink, count, work, 1, R->staging, st);
    }
    const size_t smem = sizeof(double) * (20 + 5 * R->s + 5 * R->rin);
    const int64_t n_chunks = (n + kThreads - 1) / kThreads;
    rollout_kernel<<<grid_blocks(n_chunks, 8), kThreads, smem, st>>>(R->d_data, R->s, R->rin, R->k_steps, R->input_mode,
                                                                     x, y, p, v, n, sink, first, count);
    CARMPC_CUDA(cudaGetLastError());
    return CARMPC_OK;
}

// chunked double-buffered host pipeline shared by the two *_host entry points
template <class Launch>
static int host_pipeline(HostStage& S, const double* h_x, const double* h_y, const double* h_psi, const double* h_v,
                         int64_t n, uint32_t* h_bits, int32_t* h_first, int64_t* h_count, Launch launch) {
    int rc = S.init(h_first != nullptr, n);
    if (rc != CARMPC_OK) return rc;
    const int64_t chunk = S.cap;                           // = kChunkSamples whenever the call needs more than one chunk
    CARMPC_CUDA(cudaMemsetAsync(S.d_count, 0, sizeof(unsigned long long), S.streams[0]));
    CARMPC_CUDA(cudaStreamSynchronize(S.streams[0]));
    int slot = 0;
    for (int64_t s = 0; s < n; s += chunk, slot ^= 1) {
        const int64_t len = (n - s < chunk) ? (n - s) : chunk;
        cudaStream_t st = S.streams[slot];
        double* d = S.d_coord[slot];
        const double* src[4] = {h_x, h_y, h_psi, h_v};
        for (int a = 0; a < 4; ++a)
            CARMPC_CUDA(cudaMemcpyAsync(d + a * chunk, src[a] + s, sizeof(double) * len, cudaMemcpyHostToDevice, st));
        rc = launch(d, d + chunk, d + 2 * chunk, d + 3 * chunk, len, single_sink(S.d_bits[slot]), S.d_first[slot], S.d_count,
                    S.d_work + 2 * slot, st);
        if (rc != CARMPC_OK) return rc;
        CARMPC_CUDA(cudaMemcpyAsync(h_bits + (s >> 5), S.d_bits[slot], sizeof(uint32_t) * ((len + 31) / 32),
                                    cudaMemcpyDeviceToHost, st));
        if (h_first)
            CARMPC_CUDA(cudaMemcpyAsync(h_first + s, S.d_first[slot], sizeof(int32_t) * len, cudaMemcpyDeviceToHost, st));
    }
    CARMPC_CUDA(cudaStreamSynchronize(S.streams[0]));
    CARMPC_CUDA(cudaStreamSynchronize(S.streams[1]));
    if (h_count) {
        unsigned long long c = 0;
        CARMPC_CUDA(cudaMemcpy(&c, S.d_count, sizeof(c), cudaMemcpyDeviceToHost));
        *h_count = (int64_t)c;
    }
    return CARMPC_OK;
}

// ---- profile-guided row order ------------------------------------------------------------------------------------------
// The conjunction over rows does not depend on their order, but the cost does: a warp stops as soon as every one of
// its samples is rejected.  Which rows reject most depends on where the samples lie, so the first large call runs a
// pilot over a strided subsample (every row in float64, one 64-bit "violated rows" mask per sample) and the host
// orders the rows greedily: first the row that rejects most samples, then the row that rejects most of the samples
// still alive, and so on.  Results are bit-identical for any order.
__global__ void __launch_bounds__(256)
pilot_kernel(const double* __restrict__ g_rows, int rows, const double* __restrict__ gx, const double* __restrict__ gy,
             const double* __restrict__ gp, const double* __restrict__ gv, int64_t n, int64_t stride, int n_sub,
             unsigned long long* __restrict__ masks) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n_sub) return;
    const int64_t i = (int64_t)k * stride;
    if (i >= n) { masks[k] = 0ull; return; }
    const double x = gx[i], y = gy[i], p = gp[i], v = gv[i];
    unsigned long long m = 0ull;
    for (int r = 0; r < rows; ++r) {
        const double* a = g_rows + 5 * r;
        const double lhs = fma(a[3], v, fma(a[2], p, fma(a[1], y, a[0] * x)));
        if (!(lhs <= a[4])) m |= 1ull << r;
    }
    masks[k] = m;
}

static int upload_rows(Polytope* P, cudaStream_t st) {
    const int rows = P->rows;
    std::vector<RowF32> r32(pad_rows(rows) > 0 ? pad_rows(rows) : 8);
    for (RowF32& q : r32) { q.na0 = q.na1 = q.na2 = q.na3 = 0.f; q.b = INFINITY; q.pad0 = q.pad1 = q.pad2 = 0.f; }
    for (int i = 0; i < rows; ++i) {
        const double* a = P->h_rows.data() + 5 * i;
        RowF32 q;
        q.na0 = (float)-a[0]; q.na1 = (float)-a[1]; q.na2 = (float)-a[2]; q.na3 = (float)-a[3];
        q.b = (float)a[4];
        q.pad0 = q.pad1 = q.pad2 = 0.f;
        r32[i] = q;
    }
    if (rows > 0) CARMPC_CUDA(cudaMemcpyAsync(P->d_rows, P->h_rows.data(), sizeof(double) * 5 * rows, cudaMemcpyHostToDevice, st));
    CARMPC_CUDA(cudaMemcpyAsync(P->d_rows32, r32.data(), sizeof(RowF32) * r32.size(), cudaMemcpyHostToDevice, st));
    CARMPC_CUDA(cudaStreamSynchronize(st));            // r32 / h_rows are pageable host memory
    return CARMPC_OK;
}

static int tune_row_order(Polytope* P, const double* x, const double* y, const double* p, const double* v, int64_t n,
                          cudaStream_t st) {
    const int rows = P->rows;
    P->tuned = true;
    if (rows < 2 || rows > 64 || n < 1024) return CARMPC_OK;
    const int n_sub = (int)std::min<int64_t>(1 << 16, n);
    const int64_t stride = n / n_sub;
    unsigned long long* d_masks = nullptr;
    CARMPC_CUDA(cudaMalloc(&d_masks, sizeof(unsigned long long) * n_sub));
    pilot_kernel<<<(n_sub + 255) / 256, 256, 0, st>>>(P->d_rows, rows, x, y, p, v, n, stride, n_sub, d_masks);
    std::vector<unsigned long long> masks(n_sub);
    cudaError_t err = cudaMemcpyAsync(masks.data(), d_masks, sizeof(unsigned long long) * n_sub, cudaMemcpyDeviceToHost, st);
    if (err == cudaSuccess) err = cudaStreamSynchronize(st);
    cudaFree(d_masks);
    CARMPC_CUDA(err);
    // greedy cover
    std::vector<unsigned long long> alive;
    alive.reserve(n_sub);
    for (unsigned long long m : masks) if (m) alive.push_back(m);
    std::vector<int> order;
    std::vector<char> used(rows, 0);
    while (!alive.empty() && (int)order.size() < rows) {
        int cnt[64] = {0};
        for (unsigned long long m : alive)
            for (unsigned long long t = m; t; t &= t - 1) ++cnt[__builtin_ctzll(t)];
        int best = -1;
        for (int r = 0; r < rows; ++r) if (!used[r] && (best < 0 || cnt[r] > cnt[best])) best = r;
        if (best < 0 || cnt[best] == 0) break;
        used[best] = 1;
        order.push_back(best);
        size_t w = 0;
        for (unsigned long long m : alive) if (!((m >> best) & 1ull)) alive[w++] = m;
        alive.resize(w);
    }
    for (int r = 0; r < rows; ++r) if (!used[r]) order.push_back(r);       // the rest keeps its relative order
    std::vector<double> sorted(5 * rows);
    for (int i = 0; i < rows; ++i)
        for (int k = 0; k < 5; ++k) sorted[5 * i + k] = P->h_rows[5 * order[i] + k];
    P->h_rows.swap(sorted);
    return upload_rows(P, st);
}

// The same idea for the expanded rows of the screened rollout form (up to 512 rows, float32 images: the order is a
// heuristic, the decisions do not depend on it): masks of `words` 64-bit words per subsample.
__global__ void __launch_bounds__(256)
pilot32_kernel(const RowF32* __restrict__ g_rows32, int rows, int words, const double* __restrict__ gx,
               const double* __restrict__ gy, const double* __restrict__ gp, const double* __restrict__ gv, int64_t n,
               int64_t stride, int n_sub, unsigned long long* __restrict__ masks) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n_sub) return;
    const int64_t i = (int64_t)k * stride;
    unsigned long long* out = masks + (size_t)k * words;
    for (int w = 0; w < words; ++w) out[w] = 0ull;
    if (i >= n) return;
    const float x = (float)gx[i], y = (float)gy[i], p = (float)gp[i], v = (float)gv[i];
    for (int r = 0; r < rows; ++r) {
        const RowF32 q = g_rows32[r];
        const float m = fmaf(q.na3, v, fmaf(q.na2, p, fmaf(q.na1, y, fmaf(q.na0, x, q.b))));
        if (!(m >= 0.f)) out[r >> 6] |= 1ull << (r & 63);
    }
}

static int tune_rollout_order(Rollout* R, const double* x, const double* y, const double* p, const double* v, int64_t n,
                              cudaStream_t st) {
    R->tuned = true;
    const int rows = R->rows32;
    if (rows < 2 || n < 1024 || R->d_rows32 == nullptr) return CARMPC_OK;
    const int words = (rows + 63) / 64;
    const int n_sub = (int)std::min<int64_t>(1 << 16, n);
    const int64_t stride = n / n_sub;
    unsigned long long* d_masks = nullptr;
    CARMPC_CUDA(cudaMalloc(&d_masks, sizeof(unsigned long long) * n_sub * words));
    pilot32_kernel<<<(n_sub + 255) / 256, 256, 0, st>>>(R->d_rows32, rows, words, x, y, p, v, n, stride, n_sub, d_masks);
    std::vector<unsigned long long> masks((size_t)n_sub * words);
    cudaError_t err = cudaMemcpyAsync(masks.data(), d_masks, sizeof(unsigned long long) * masks.size(), cudaMemcpyDeviceToHost, st);
    if (err == cudaSuccess) err = cudaStreamSynchronize(st);
    cudaFree(d_masks);
    CARMPC_CUDA(err);
    // greedy cover: the row that rejects most of the subsamples still alive comes next
    std::vector<int> alive;
    alive.reserve(n_sub);
    for (int k = 0; k < n_sub; ++k) {
        bool any = false;
        for (int w = 0; w < words; ++w) any = any || masks[(size_t)k * words + w] != 0ull;
        if (any) alive.push_back(k);
    }
    std::vector<int> order;
    std::vector<char> used(rows, 0);
    std::vector<int> cnt(rows);
    while (!alive.empty() && (int)order.size() < rows) {
        std::fill(cnt.begin(), cnt.end(), 0);
        for (int k : alive)
            for (int w = 0; w < words; ++w)
                for (unsigned long long t = masks[(size_t)k * words + w]; t; t &= t - 1) ++cnt[64 * w + __builtin_ctzll(t)];
        int best = -1;
        for (int r = 0; r < rows; ++r) if (!used[r] && (best < 0 || cnt[r] > cnt[best])) best = r;
        if (best < 0 || cnt[best] == 0) break;
        used[best] = 1;
        order.push_back(best);
        size_t w = 0;
        for (int k : alive) if (!((masks[(size_t)k * words + (best >> 6)] >> (best & 63)) & 1ull)) alive[w++] = k;
        alive.resize(w);
    }
    for (int r = 0; r < rows; ++r) if (!used[r]) order.push_back(r);       // the rest keeps its relative order
    std::vector<RowF32> sorted(R->h_rows32);
    for (int i = 0; i < rows; ++i) sorted[i] = R->h_rows32[order[i]];
    R->h_rows32.swap(sorted);
    CARMPC_CUDA(cudaMemcpyAsync(R->d_rows32, R->h_rows32.data(), sizeof(RowF32) * R->h_rows32.size(), cudaMemcpyHostToDevice, st));
    CARMPC_CUDA(cudaStreamSynchronize(st));
    return CARMPC_OK;
}

}  // namespace carmpc

using namespace carmpc;

extern "C" {

int carmpc_polytope_create(const double* h_Ab, int rows, void** handle) {
    CARMPC_REQUIRE(h_Ab != nullptr && handle != nullptr, "null pointer");
    CARMPC_REQUIRE(rows >= 0 && rows <= kMaxRows, "rows must be in [0, 512]");
    Polytope* P = new Polytope();
    P->kind = kPolytope;
    P->rows = rows;
    cudaGetDevice(&P->device);
    // sort the rows by sparsity pattern: fewest non-zeros first (cheapest, and for these sets the axis-aligned
    // bounds that reject most samples), stable within a pattern
    std::vector<int> order(rows), pat(rows);
    for (int r = 0; r < rows; ++r) {
        order[r] = r;
        int m = 0;
        for (int k = 0; k < 4; ++k) {
            if (isnan(h_Ab[5 * r + k]) || isinf(h_Ab[5 * r + k])) { delete P; set_error("carmpc_polytope_create: non-finite coefficient in row %d", r); return CARMPC_ERR_INVALID; }
            if (h_Ab[5 * r + k] != 0.0) m |= 1 << k;
        }
        if (isnan(h_Ab[5 * r + 4])) { delete P; set_error("carmpc_polytope_create: NaN bound in row %d", r); return CARMPC_ERR_INVALID; }
        pat[r] = m;
    }
    auto popc = [](int m) { return (m & 1) + ((m >> 1) & 1) + ((m >> 2) & 1) + ((m >> 3) & 1); };
    std::stable_sort(order.begin(), order.end(), [&](int a, int b) {
        if (popc(pat[a]) != popc(pat[b])) return popc(pat[a]) < popc(pat[b]);
        return pat[a] < pat[b];
    });
    std::vector<double> sorted(5 * (rows > 0 ? rows : 1), 0.0);
    std::vector<RowF32> r32(pad_rows(rows) > 0 ? pad_rows(rows) : 8);
    for (RowF32& q : r32) { q.na0 = q.na1 = q.na2 = q.na3 = 0.f; q.b = INFINITY; q.pad0 = q.pad1 = q.pad2 = 0.f; }
    double l1max = 0.0, bmax = 0.0;
    bool faithful = true;            // every coefficient and every finite b has a finite float32 image
    for (int i = 0; i < rows; ++i) {
        const double* a = h_Ab + 5 * order[i];
        for (int k = 0; k < 5; ++k) sorted[5 * i + k] = a[k];
        RowF32 q;
        q.na0 = (float)-a[0]; q.na1 = (float)-a[1]; q.na2 = (float)-a[2]; q.na3 = (float)-a[3];
        q.b = (float)a[4];
        q.pad0 = q.pad1 = q.pad2 = 0.f;
        r32[i] = q;
        faithful = faithful && std::isfinite(q.na0) && std::isfinite(q.na1) && std::isfinite(q.na2) && std::isfinite(q.na3) &&
                   (isinf(a[4]) || std::isfinite(q.b));
        l1max = std::max(l1max, fabs(a[0]) + fabs(a[1]) + fabs(a[2]) + fabs(a[3]));
        if (!isinf(a[4])) bmax = std::max(bmax, fabs(a[4]));
    }
    // Rounding-error bound of the float32 margin  m = fma(-a3, v, fma(-a2, psi, fma(-a1, y, fma(-a0, x, b))))  against the
    // exact  b - a . p , as long as no float32 value in it overflows:
    //   - b, the coefficients and the coordinates are rounded once to float32 (relative 2^-24), and each of the <= 4 fmas
    //     rounds once (relative 2^-24 of an intermediate, which is at most |b| + sum |a_k| |p_k| up to O(2^-24)), so
    //     |error| <= (4 + 2 + 1) 2^-24 (|b| + sum |a_k| |p_k|) (1 + O(2^-24));
    //   - below the normal range a rounding is off by up to 2^-150 in absolute terms instead: for b, a coefficient or an fma
    //     result that costs at most 2^-150 (4 + |p|_1), inside the 1e-37 floors; for a coordinate (subnormal or zero in
    //     float32) it costs |a_k| 2^-150 each, at most l1max 2^-150 in all: the l1max 2^-149 term of beta0;
    //   - the float64 chain's own error (2^-51 of the same magnitude) is covered by using 8 instead of 7 and by rounding the
    //     two constants up.
    // The no-overflow condition is enforced, not assumed.  A polytope whose coefficients or finite bounds have no finite
    // float32 image, or whose constants reach 1e30, gets an infinite beta pair: no sample is decided in float32 and mode 1
    // returns what the float64 chain returns for every sample.  Otherwise screen32 leaves every sample whose bound exceeds
    // kScreenMaxBound (non-finite and huge coordinates among them) to the float64 chain.  Rows with b = +inf stay on the
    // screen: their float32 margin is exactly +inf, which is right.
    const double u8 = 8.0 * 5.9604644775390625e-08, tiny = 1.401298464324817e-45;      // 2^-149
    const double b0 = u8 * bmax * 1.000001 + l1max * tiny + 1e-37, b1 = u8 * l1max * 1.000001 + 1e-37;
    if (faithful && b0 < 1e30 && b1 < 1e30) {
        P->beta0 = nextafterf((float)b0, INFINITY);
        P->beta1 = nextafterf((float)b1, INFINITY);
    } else {
        P->beta0 = P->beta1 = INFINITY;
    }
    P->h_rows = sorted;
    h_Ab = sorted.data();
    auto fail = [&](int code) { delete P; return code; };
    if (cudaMalloc(&P->d_rows, sizeof(double) * 5 * (rows > 0 ? rows : 1)) != cudaSuccess ||
        cudaMalloc(&P->d_rows32, sizeof(RowF32) * r32.size()) != cudaSuccess ||
        cudaMalloc(&P->d_work, sizeof(unsigned long long) * 2) != cudaSuccess ||
        cudaMemset(P->d_work, 0, sizeof(unsigned long long) * 2) != cudaSuccess) {
        set_error("carmpc_polytope_create: cudaMalloc failed: %s", cudaGetErrorString(cudaGetLastError()));
        return fail(CARMPC_ERR_CUDA);
    }
    if (rows > 0) {
        if (cudaMemcpy(P->d_rows, h_Ab, sizeof(double) * 5 * rows, cudaMemcpyHostToDevice) != cudaSuccess ||
            cudaMemcpy(P->d_rows32, r32.data(), sizeof(RowF32) * r32.size(), cudaMemcpyHostToDevice) != cudaSuccess) {
            set_error("carmpc_polytope_create: cudaMemcpy failed: %s", cudaGetErrorString(cudaGetLastError()));
            return fail(CARMPC_ERR_CUDA);
        }
    }
    *handle = P;
    return CARMPC_OK;
}

int carmpc_membership_bitset(void* polytope, const double* d_x, const double* d_y, const double* d_psi,
                             const double* d_v, int64_t n, uint32_t* d_bits, int64_t* d_count, int mode,
                             void* stream) {
    Polytope* P = check_handle<Polytope>(polytope, kPolytope);
    CARMPC_REQUIRE(P != nullptr, "not a polytope handle");
    CARMPC_REQUIRE(n >= 0, "n");
    CARMPC_REQUIRE(mode == 0 || mode == 1, "mode must be 0 or 1");
    if (n == 0) {
        if (d_count) CARMPC_CUDA(cudaMemsetAsync(d_count, 0, sizeof(int64_t), (cudaStream_t)stream));
        return CARMPC_OK;
    }
    CARMPC_REQUIRE(d_x && d_y && d_psi && d_v && d_bits, "null device pointer");
    cudaStream_t st = (cudaStream_t)stream;
    if (!P->tuned && n >= ((int64_t)1 << 20)) {
        const int rc = tune_row_order(P, d_x, d_y, d_psi, d_v, n, st);
        if (rc != CARMPC_OK) return rc;
    }
    if (d_count) CARMPC_CUDA(cudaMemsetAsync(d_count, 0, sizeof(int64_t), st));
    return launch_membership(P, d_x, d_y, d_psi, d_v, n, single_sink(d_bits), reinterpret_cast<unsigned long long*>(d_count),
                             P->d_work, mode, st);
}

int carmpc_polytope_tune(void* polytope, const double* d_x, const double* d_y, const double* d_psi, const double* d_v,
                         int64_t n, void* stream) {
    Polytope* P = check_handle<Polytope>(polytope, kPolytope);
    CARMPC_REQUIRE(P != nullptr, "not a polytope handle");
    CARMPC_REQUIRE(n >= 0, "n");
    if (n == 0) return CARMPC_OK;
    CARMPC_REQUIRE(d_x && d_y && d_psi && d_v, "null device pointer");
    return tune_row_order(P, d_x, d_y, d_psi, d_v, n, (cudaStream_t)stream);
}

int carmpc_membership_grid(void* polytope, const double* h_axes, const int32_t dims[4],
                           const int32_t axis_to_state[4], uint32_t* d_bits, int64_t* d_count, void* stream) {
    Polytope* P = check_handle<Polytope>(polytope, kPolytope);
    CARMPC_REQUIRE(P != nullptr, "not a polytope handle");
    CARMPC_REQUIRE(h_axes && dims && axis_to_state && d_bits, "null pointer");
    GridDesc gd;
    int64_t n = 1;
    int off = 0, seen = 0;
    for (int k = 0; k < 4; ++k) {
        CARMPC_REQUIRE(dims[k] >= 1 && dims[k] <= 4096, "each axis must have 1..4096 points");
        CARMPC_REQUIRE(axis_to_state[k] >= 0 && axis_to_state[k] < 4, "axis_to_state entries must be 0..3");
        seen |= 1 << axis_to_state[k];
        gd.dims[k] = dims[k];
        gd.state_of_axis[k] = axis_to_state[k];
        gd.offset[k] = off;
        off += dims[k];
        n *= dims[k];
    }
    CARMPC_REQUIRE(seen == 15, "axis_to_state must be a permutation of 0..3");
    cudaStream_t st = (cudaStream_t)stream;
    if (P->d_axes == nullptr) {
        CARMPC_CUDA(cudaMalloc(&P->d_axes, sizeof(double) * 4 * 4096));
        CARMPC_CUDA(cudaMallocHost(&P->h_axes, sizeof(double) * 4 * 4096));
    }
    CARMPC_CUDA(cudaStreamSynchronize(st));            // the staging copy of a previous call must have been consumed
    for (int i = 0; i < off; ++i) P->h_axes[i] = h_axes[i];
    double* d_axes = P->d_axes;
    CARMPC_CUDA(cudaMemcpyAsync(d_axes, P->h_axes, sizeof(double) * off, cudaMemcpyHostToDevice, st));
    if (!P->tuned && n >= ((int64_t)1 << 20)) {
        // profile-guided row order from a strided subsample of the grid, expanded on the host (65,536 points, once per polytope)
        const int n_sub = 1 << 16;
        const int64_t stride = n / n_sub;
        std::vector<double> sub((size_t)4 * n_sub);
        for (int k = 0; k < n_sub; ++k) {
            int64_t rem = (int64_t)k * stride;
            for (int ax = 3; ax >= 0; --ax) {
                const int64_t q = rem / dims[ax];
                sub[(size_t)axis_to_state[ax] * n_sub + k] = h_axes[gd.offset[ax] + (int)(rem - q * dims[ax])];
                rem = q;
            }
        }
        double* d_sub = nullptr;
        CARMPC_CUDA(cudaMalloc(&d_sub, sizeof(double) * 4 * n_sub));
        cudaError_t err = cudaMemcpyAsync(d_sub, sub.data(), sizeof(double) * 4 * n_sub, cudaMemcpyHostToDevice, st);
        int rc = CARMPC_OK;
        if (err == cudaSuccess) rc = tune_row_order(P, d_sub, d_sub + n_sub, d_sub + 2 * n_sub, d_sub + 3 * n_sub, n_sub, st);
        cudaStreamSynchronize(st);
        cudaFree(d_sub);
        CARMPC_CUDA(err);
        if (rc != CARMPC_OK) return rc;
    }
    if (d_count) CARMPC_CUDA(cudaMemsetAsync(d_count, 0, sizeof(int64_t), st));
    const size_t smem = membership_smem(P->rows) + (sizeof(double) + sizeof(float)) * off;
    CARMPC_CUDA(cudaFuncSetAttribute(membership_grid_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int64_t n_chunks = (n + kChunk - 1) / kChunk;
    membership_grid_kernel<<<grid_blocks(n_chunks, 4), kThreads, smem, st>>>(
        P->d_rows, P->d_rows32, P->rows, pad_rows(P->rows), screen_const(P), d_axes, gd, n, d_bits,
        reinterpret_cast<unsigned long long*>(d_count));
    CARMPC_CUDA(cudaGetLastError());
    return CARMPC_OK;
}

int carmpc_membership_bitset_host(void* polytope, const double* h_x, const double* h_y, const double* h_psi,
                                  const double* h_v, int64_t n, uint32_t* h_bits, int64_t* h_count, int mode) {
    Polytope* P = check_handle<Polytope>(polytope, kPolytope);
    CARMPC_REQUIRE(P != nullptr, "not a polytope handle");
    CARMPC_REQUIRE(n >= 0, "n");
    CARMPC_REQUIRE(mode == 0 || mode == 1, "mode must be 0 or 1");
    if (h_count) *h_count = 0;
    if (n == 0) return CARMPC_OK;
    CARMPC_REQUIRE(h_x && h_y && h_psi && h_v && h_bits, "null host pointer");
    return host_pipeline(P->stage, h_x, h_y, h_psi, h_v, n, h_bits, nullptr, h_count,
                         [&](const double* x, const double* y, const double* p, const double* v, int64_t len,
                             const BitSink& bits, int32_t*, unsigned long long* count, unsigned long long* work, cudaStream_t st) {
                             return launch_membership(P, x, y, p, v, len, bits, count, work, mode, st);
                         });
}

int carmpc_rollout_create(const double* h_Ak, const double* h_Acon, const double* h_bcon, int s,
                          const double* h_Ain, const double* h_bin, int rin, const double* h_goal,
                          int k_steps, int input_check_mode, void** handle) {
    CARMPC_REQUIRE(h_Ak && h_goal && handle, "null pointer");
    CARMPC_REQUIRE(s >= 0 && s <= 256 && rin >= 0 && rin <= 256, "row counts must be in [0, 256]");
    CARMPC_REQUIRE((s == 0 || (h_Acon && h_bcon)) && (rin == 0 || (h_Ain && h_bin)), "null row pointer");
    CARMPC_REQUIRE(k_steps >= 0 && k_steps <= 100000, "k_steps");
    CARMPC_REQUIRE(input_check_mode == 0 || input_check_mode == 1, "input_check_mode must be 0 or 1");
    std::vector<double> data(20 + 5 * s + 5 * rin);
    for (int i = 0; i < 16; ++i) data[i] = h_Ak[i];
    for (int i = 0; i < 4; ++i) data[16 + i] = h_goal[i];
    double* q = data.data() + 20;
    for (int i = 0; i < 4 * s; ++i) *q++ = h_Acon[i];
    for (int i = 0; i < s; ++i) *q++ = h_bcon[i];
    for (int i = 0; i < 4 * rin; ++i) *q++ = h_Ain[i];
    for (int i = 0; i < rin; ++i) *q++ = h_bin[i];
    Rollout* R = new Rollout();
    R->kind = kRollout;
    R->s = s; R->rin = rin; R->k_steps = k_steps; R->input_mode = input_check_mode;
    cudaGetDevice(&R->device);
    if (cudaMalloc(&R->d_data, sizeof(double) * data.size()) != cudaSuccess ||
        cudaMalloc(&R->d_work, sizeof(unsigned long long) * 2) != cudaSuccess ||
        cudaMemset(R->d_work, 0, sizeof(unsigned long long) * 2) != cudaSuccess ||
        cudaMemcpy(R->d_data, data.data(), sizeof(double) * data.size(), cudaMemcpyHostToDevice) != cudaSuccess) {
        set_error("carmpc_rollout_create: %s", cudaGetErrorString(cudaGetLastError()));
        delete R;
        return CARMPC_ERR_CUDA;
    }
    // Float32 screen.  The row value at step t is linear in the sample: a_r A_k^t (p - goal) <= b_r, so the rollout is
    // a membership test against the expanded rows g = a_r A_k^t, b' = b_r + g . goal (absolute coordinates).  They are
    // built here in long double, stored as float32 and evaluated like the H-rep screen; a sample is decided by the
    // screen only when its smallest margin clears the bound
    //     8 u32 (|b'| + sum |g_k| |p_k|)   float32 evaluation (as for the H-rep rows)
    //   + l1max 2^-149                     coordinates below float32's normal range (as for the H-rep rows)
    //   + c64 G (sum |p_k| + |goal|_1)     float64 step-by-step rollout vs the exact linear functional, with
    //                                      G = max entry of |a_r| |A_k|^t and c64 = 16 (k + 3) 2^-53,
    // everything else is re-evaluated by the float64 contract chain (rollout64).  As for the H-rep rows the bound needs the
    // float32 chain not to overflow: the screen is built only when every expanded row has a finite float32 image and both
    // constants stay below 1e30, and screen32 decides no sample whose bound exceeds kScreenMaxBound.
    const long total_rows = (long)s * (k_steps + 1) + (long)rin * (input_check_mode == 1 ? k_steps + 1 : 1);
    if (total_rows > 0 && total_rows <= kMaxRows) {
        std::vector<RowF32> r32(pad_rows((int)total_rows));
        for (RowF32& q : r32) { q.na0 = q.na1 = q.na2 = q.na3 = 0.f; q.b = INFINITY; q.pad0 = q.pad1 = q.pad2 = 0.f; }
        long double M[16], Mabs[16];
        for (int i = 0; i < 16; ++i) M[i] = Mabs[i] = (i % 5 == 0) ? 1.0L : 0.0L;
        long double l1max = 0, bmax = 0, gabs_max = 0, goal1 = 0;
        for (int k = 0; k < 4; ++k) goal1 += fabsl((long double)h_goal[k]);
        bool finite = true;
        int w = 0;
        auto emit = [&](const double* a, double b) {
            long double g[4], ga[4], bp = b, l1 = 0;
            for (int j = 0; j < 4; ++j) {
                g[j] = ga[j] = 0;
                for (int i = 0; i < 4; ++i) { g[j] += (long double)a[i] * M[4 * i + j]; ga[j] += fabsl((long double)a[i]) * Mabs[4 * i + j]; }
                bp += g[j] * (long double)h_goal[j];
                l1 += fabsl(g[j]);
                gabs_max = std::max(gabs_max, ga[j]);
            }
            RowF32 q;
            q.na0 = (float)-g[0]; q.na1 = (float)-g[1]; q.na2 = (float)-g[2]; q.na3 = (float)-g[3];
            q.b = (float)bp;
            q.pad0 = q.pad1 = q.pad2 = 0.f;
            for (int j = 0; j < 4; ++j) R->h_rows64.push_back((double)g[j]);
            R->h_rows64.push_back(b == INFINITY ? INFINITY : (double)bp);
            finite = finite && std::isfinite(q.na0) && std::isfinite(q.na1) && std::isfinite(q.na2) && std::isfinite(q.na3) &&
                     (std::isinf(b) || std::isfinite(q.b));
            if (b == INFINITY) q.b = INFINITY;
            r32[w++] = q;
            l1max = std::max(l1max, l1);
            if (std::isfinite((double)bp)) bmax = std::max(bmax, fabsl(bp));
        };
        for (int t = 0; t <= k_steps; ++t) {
            for (int r = 0; r < s; ++r) emit(h_Acon + 4 * r, h_bcon[r]);
            if (t == 0 || input_check_mode == 1)
                for (int r = 0; r < rin; ++r) emit(h_Ain + 4 * r, h_bin[r]);
            long double N[16], Na[16];
            for (int i = 0; i < 4; ++i)
                for (int j = 0; j < 4; ++j) {
                    N[4 * i + j] = Na[4 * i + j] = 0;
                    for (int l = 0; l < 4; ++l) {
                        N[4 * i + j] += (long double)h_Ak[4 * i + l] * M[4 * l + j];
                        Na[4 * i + j] += fabsl((long double)h_Ak[4 * i + l]) * Mabs[4 * l + j];
                    }
                }
            for (int i = 0; i < 16; ++i) { M[i] = N[i]; Mabs[i] = Na[i]; }
        }
        const long double u8 = 8.0L * 5.9604644775390625e-08L, c64 = 16.0L * (k_steps + 3) * 1.1102230246251565e-16L;
        const long double tiny = 1.401298464324817e-45L;                                   // 2^-149: coordinates below float32's normal range
        const long double b0 = u8 * bmax * 1.000001L + l1max * tiny + c64 * gabs_max * goal1 + 1e-37L,
                          b1 = u8 * l1max * 1.000001L + c64 * gabs_max + 1e-37L;
        if (finite && std::isfinite((double)b0) && std::isfinite((double)b1) && (double)b0 < 1e30 && (double)b1 < 1e30) {
            R->beta0 = nextafterf((float)b0, INFINITY);
            R->beta1 = nextafterf((float)b1, INFINITY);
            R->in0 = R->beta0;
            R->in1 = R->beta1;
            R->rows_padded = (int)r32.size();
            R->rows32 = (int)total_rows;
            R->h_rows32 = r32;
            if (cudaMalloc(&R->d_rows32, sizeof(RowF32) * r32.size()) != cudaSuccess ||
                cudaMemcpy(R->d_rows32, r32.data(), sizeof(RowF32) * r32.size(), cudaMemcpyHostToDevice) != cudaSuccess) {
                set_error("carmpc_rollout_create: %s", cudaGetErrorString(cudaGetLastError()));
                delete R;
                return CARMPC_ERR_CUDA;
            }
        }
    }
    *handle = R;
    return CARMPC_OK;
}

int carmpc_rollout_get_rows(void* rollout, double* h_rows, int capacity) {
    Rollout* R = check_handle<Rollout>(rollout, kRollout);
    CARMPC_REQUIRE(R != nullptr, "not a rollout handle");
    const int cnt = (int)R->h_rows64.size();
    if (h_rows) {
        CARMPC_REQUIRE(capacity >= cnt, "capacity too small");
        memcpy(h_rows, R->h_rows64.data(), sizeof(double) * cnt);
    }
    return R->d_rows32 != nullptr ? cnt / 5 : 0;
}

int carmpc_rollout_reduce_screen(void* rollout, const int32_t* h_kept, int n_kept, const int32_t* h_dual_idx,
                                 const double* h_dual_w, int n_dual) {
    Rollout* R = check_handle<Rollout>(rollout, kRollout);
    CARMPC_REQUIRE(R != nullptr, "not a rollout handle");
    CARMPC_REQUIRE(R->d_rows32 != nullptr, "this rollout has no float32 screen");
    const int rows = (int)R->h_rows64.size() / 5;
    CARMPC_REQUIRE(h_kept && n_kept >= 1 && n_kept <= rows, "kept rows");
    CARMPC_REQUIRE(n_kept == rows || (h_dual_idx && h_dual_w && n_dual >= 1 && n_dual <= 16), "dual certificates");
    std::vector<char> kept(rows, 0);
    for (int i = 0; i < n_kept; ++i) {
        CARMPC_REQUIRE(h_kept[i] >= 0 && h_kept[i] < rows && !kept[h_kept[i]], "kept row index out of range or repeated");
        kept[h_kept[i]] = 1;
    }
    // Every dropped row d needs a certificate lambda >= 0 over kept rows with  g_d ~ sum lambda_k g_k  and
    // sum lambda_k b_k <~ b_d : then, with M_r(p) = b_r - g_r . p,
    //     M_d >= sum lambda_k M_k - tol_d - rho_d |p|_1 ,   tol_d = (sum lambda_k b_k - b_d)+ ,  rho_d = |g_d - sum lambda_k g_k|_inf
    // so a sample whose smallest float32 margin over the KEPT rows exceeds
    //     beta(p) max(1, 1 / L) + (tol + rho |p|_1) / L ,    L = min_d sum lambda_k
    // clears the float64 band of every dropped row as well.  The certificates are only CHECKED here (in long double, against
    // the rows this handle built), wherever they come from; what they do not prove widens the band or is refused.
    long double lam_min = INFINITY, tol_max = 0, rho_max = 0;
    const double* G = R->h_rows64.data();
    for (int d = 0; d < rows; ++d) {
        if (kept[d]) continue;
        if (G[5 * d + 4] == INFINITY) continue;                 // a row without a bound constrains nothing
        long double sum = 0, bsum = 0, acc[4] = {0, 0, 0, 0};
        for (int j = 0; j < n_dual; ++j) {
            const int k = h_dual_idx[(size_t)d * n_dual + j];
            const long double w = h_dual_w[(size_t)d * n_dual + j];
            if (w == 0) continue;
            CARMPC_REQUIRE(k >= 0 && k < rows && kept[k] && w > 0 && std::isfinite((double)w) && G[5 * k + 4] != INFINITY,
                           "a certificate must combine kept rows with non-negative weights");
            sum += w;
            bsum += w * (long double)G[5 * k + 4];
            for (int c = 0; c < 4; ++c) acc[c] += w * (long double)G[5 * k + c];
        }
        CARMPC_REQUIRE(sum > 1e-9L, "empty certificate for a dropped row");
        long double rho = 0;
        for (int c = 0; c < 4; ++c) rho = std::max(rho, fabsl((long double)G[5 * d + c] - acc[c]));
        lam_min = std::min(lam_min, sum);
        tol_max = std::max(tol_max, bsum - (long double)G[5 * d + 4]);
        rho_max = std::max(rho_max, rho);
    }
    long double in0 = R->beta0, in1 = R->beta1;
    if (lam_min != INFINITY) {
        const long double scale = std::max(1.0L, 1.0L / lam_min);
        in0 = (long double)R->beta0 * scale + tol_max / lam_min;
        in1 = (long double)R->beta1 * scale + rho_max / lam_min;
    }
    CARMPC_REQUIRE(std::isfinite((double)in0) && std::isfinite((double)in1) && (double)in0 < 1e-2 && (double)in1 < 1e-2,
                   "the certificates leave an acceptance band wider than 1e-2: screen not reduced");
    std::vector<RowF32> r32(pad_rows(n_kept));
    for (RowF32& q : r32) { q.na0 = q.na1 = q.na2 = q.na3 = 0.f; q.b = INFINITY; q.pad0 = q.pad1 = q.pad2 = 0.f; }
    for (int i = 0; i < n_kept; ++i) {
        const double* g = G + 5 * (size_t)h_kept[i];
        RowF32 q;
        q.na0 = (float)-g[0]; q.na1 = (float)-g[1]; q.na2 = (float)-g[2]; q.na3 = (float)-g[3];
        q.b = g[4] == INFINITY ? INFINITY : (float)g[4];
        q.pad0 = q.pad1 = q.pad2 = 0.f;
        r32[i] = q;
    }
    CARMPC_REQUIRE(r32.size() <= R->h_rows32.size(), "internal: the reduced screen cannot be larger than the full one");
    CARMPC_CUDA(cudaDeviceSynchronize());
    CARMPC_CUDA(cudaMemcpy(R->d_rows32, r32.data(), sizeof(RowF32) * r32.size(), cudaMemcpyHostToDevice));
    R->h_rows32 = r32;
    R->rows_padded = (int)r32.size();
    R->rows32 = n_kept;
    R->in0 = nextafterf((float)in0, INFINITY);
    R->in1 = nextafterf((float)in1, INFINITY);
    R->tuned = false;
    return CARMPC_OK;
}

int carmpc_rollout_bitset(void* rollout, const double* d_x, const double* d_y, const double* d_psi,
                          const double* d_v, int64_t n, uint32_t* d_bits, int32_t* d_first_violation,
                          int64_t* d_count, void* stream) {
    Rollout* R = check_handle<Rollout>(rollout, kRollout);
    CARMPC_REQUIRE(R != nullptr, "not a rollout handle");
    CARMPC_REQUIRE(n >= 0, "n");
    cudaStream_t st = (cudaStream_t)stream;
    if (d_count) CARMPC_CUDA(cudaMemsetAsync(d_count, 0, sizeof(int64_t), st));
    if (n == 0) return CARMPC_OK;
    CARMPC_REQUIRE(d_x && d_y && d_psi && d_v && d_bits, "null device pointer");
    if (!R->tuned && d_first_violation == nullptr && n >= ((int64_t)1 << 20)) {
        const int rc = tune_rollout_order(R, d_x, d_y, d_psi, d_v, n, st);
        if (rc != CARMPC_OK) return rc;
    }
    return launch_rollout(R, d_x, d_y, d_psi, d_v, n, single_sink(d_bits), d_first_violation,
                          reinterpret_cast<unsigned long long*>(d_count), R->d_work, st);
}

int carmpc_rollout_bitset_host(void* rollout, const double* h_x, const double* h_y, const double* h_psi,
                               const double* h_v, int64_t n, uint32_t* h_bits, int32_t* h_first_violation,
                               int64_t* h_count) {
    Rollout* R = check_handle<Rollout>(rollout, kRollout);
    CARMPC_REQUIRE(R != nullptr, "not a rollout handle");
    CARMPC_REQUIRE(n >= 0, "n");
    if (h_count) *h_count = 0;
    if (n == 0) return CARMPC_OK;
    CARMPC_REQUIRE(h_x && h_y && h_psi && h_v && h_bits, "null host pointer");
    return host_pipeline(R->stage, h_x, h_y, h_psi, h_v, n, h_bits, h_first_violation, h_count,
                         [&](const double* x, const double* y, const double* p, const double* v, int64_t len,
                             const BitSink& bits, int32_t* first, unsigned long long* count, unsigned long long* work, cudaStream_t st) {
                             return launch_rollout(R, x, y, p, v, len, bits, h_first_violation ? first : nullptr, count,
                                                   work, st);
                         });
}

// ---- sharded scans: the all-gather of the bitsets is fused into the scan kernel (shard.cuh) ------------------------------
static int shard_sink(ShardWindow* W, int64_t n_local, int64_t first_sample, int64_t group_stride, BitSink* sink,
                      unsigned long long* step_out) {
    CARMPC_REQUIRE(W->connected, "the shard window is not connected to its peers (carmpc_shard_connect)");
    CARMPC_REQUIRE(n_local >= 0 && first_sample >= 0 && group_stride >= 1, "n_local, first_sample, group_stride");
    CARMPC_REQUIRE(n_local == 0 || (first_sample & 31) == 0, "a shard starts on a whole bitset word");
    CARMPC_REQUIRE(n_local == 0 || group_stride == 1 || (first_sample & 1023) == 0, "strided shards start on a whole 1024-sample group");
    if (n_local > 0) {
        // last sample of the shard in the numbering of the whole set
        const int64_t last_local = n_local - 1;
        const int64_t last = first_sample + (last_local >> 10) * group_stride * 1024 + (last_local & 1023);
        CARMPC_REQUIRE(last < W->n_total, "the shard exceeds the sample set of the window");
    }
    const unsigned long long step = W->step + 1;
    sink->n = W->world;
    sink->stride = group_stride;
    sink->step = W->d_local_count + 3;
    sink->slot_words = W->words_pad;
    for (int r = 0; r < W->world; ++r) sink->dst[r] = W->bits(r, 0) + (first_sample >> 5);
    *step_out = step;
    return CARMPC_OK;
}

int carmpc_membership_bitset_sharded(void* polytope, void* shard, const double* d_x, const double* d_y, const double* d_psi,
                                     const double* d_v, int64_t n_local, int64_t first_sample, int64_t group_stride, int mode,
                                     int64_t* d_total_count, int defer_wait, void* stream) {
    Polytope* P = check_handle<Polytope>(polytope, kPolytope);
    CARMPC_REQUIRE(P != nullptr, "not a polytope handle");
    ShardWindow* W = check_handle<ShardWindow>(shard, kShard);
    CARMPC_REQUIRE(W != nullptr, "not a shard window");
    CARMPC_REQUIRE(mode == 0 || mode == 1, "mode must be 0 or 1");
    CARMPC_REQUIRE(n_local == 0 || (d_x && d_y && d_psi && d_v), "null device pointer");
    BitSink sink{};
    unsigned long long step = 0;
    int rc = shard_sink(W, n_local, first_sample, group_stride, &sink, &step);
    if (rc != CARMPC_OK) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    if (!P->tuned && n_local >= ((int64_t)1 << 20)) {
        rc = tune_row_order(P, d_x, d_y, d_psi, d_v, n_local, st);
        if (rc != CARMPC_OK) return rc;
    }
    rc = launch_membership(P, d_x, d_y, d_psi, d_v, n_local, sink, W->d_local_count, W->d_local_count + 1, mode, st);
    if (rc != CARMPC_OK) return rc;
    CARMPC_REQUIRE(!W->pending, "the previous step of this window was published but never waited for (carmpc_shard_wait)");
    rc = shard_publish_launch(W, st);
    if (rc != CARMPC_OK) return rc;
    if (!defer_wait) {
        rc = shard_wait_launch(W, d_total_count, st);
        if (rc != CARMPC_OK) return rc;
    }
    W->step = step;                 // (calls made through this library; graph replays advance only the device counter)
    return CARMPC_OK;
}

int carmpc_rollout_bitset_sharded(void* rollout, void* shard, const double* d_x, const double* d_y, const double* d_psi,
                                  const double* d_v, int64_t n_local, int64_t first_sample, int64_t group_stride,
                                  int64_t* d_total_count, int defer_wait, void* stream) {
    Rollout* R = check_handle<Rollout>(rollout, kRollout);
    CARMPC_REQUIRE(R != nullptr, "not a rollout handle");
    ShardWindow* W = check_handle<ShardWindow>(shard, kShard);
    CARMPC_REQUIRE(W != nullptr, "not a shard window");
    CARMPC_REQUIRE(n_local == 0 || (d_x && d_y && d_psi && d_v), "null device pointer");
    BitSink sink{};
    unsigned long long step = 0;
    int rc = shard_sink(W, n_local, first_sample, group_stride, &sink, &step);
    if (rc != CARMPC_OK) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    if (!R->tuned && n_local >= ((int64_t)1 << 20)) {
        rc = tune_rollout_order(R, d_x, d_y, d_psi, d_v, n_local, st);
        if (rc != CARMPC_OK) return rc;
    }
    rc = launch_rollout(R, d_x, d_y, d_psi, d_v, n_local, sink, nullptr, W->d_local_count, W->d_local_count + 1, st);
    if (rc != CARMPC_OK) return rc;
    CARMPC_REQUIRE(!W->pending, "the previous step of this window was published but never waited for (carmpc_shard_wait)");
    rc = shard_publish_launch(W, st);
    if (rc != CARMPC_OK) return rc;
    if (!defer_wait) {
        rc = shard_wait_launch(W, d_total_count, st);
        if (rc != CARMPC_OK) return rc;
    }
    W->step = step;
    return CARMPC_OK;
}

int carmpc_scan_staging(void* handle, int threads_per_cta, int ring_slots, int tiles_per_slot) {
    Staging g;
    g.threads = threads_per_cta; g.stages = ring_slots; g.tps = tiles_per_slot;
    if (!staging_supported(g)) {
        set_error("carmpc_scan_staging: geometry %d/%d/%d is not built into the library", threads_per_cta, ring_slots, tiles_per_slot);
        return CARMPC_ERR_UNSUPPORTED;
    }
    if (Polytope* P = check_handle<Polytope>(handle, kPolytope)) { P->staging = g; return CARMPC_OK; }
    if (Rollout* R = check_handle<Rollout>(handle, kRollout)) { R->staging = g; return CARMPC_OK; }
    set_error("carmpc_scan_staging: not a polytope or rollout handle");
    return CARMPC_ERR_INVALID;
}

}  // extern "C"
