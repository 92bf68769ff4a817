// Philox4x64-10 (Salmon et al., "Parallel random numbers: as easy as 1, 2, 3", SC 2011; the Random123 constants) and the
// Box-Muller step of the closed loops' noise.  Written out here rather than taken from cuRAND so that the exact conversion
// from counter to normal deviates is stated in one place and can be restated bit for bit (tests/noise_oracle.py;
// numpy.random.Philox is the same generator).
#pragma once

#include <stdint.h>

namespace carmpc {

struct Philox4x64 { uint64_t x[4]; };

// ten rounds on counter (c0, c1, c2, c3) with key (k0, k1); the key is bumped by the Weyl constants before rounds 1..9
__device__ __forceinline__ Philox4x64 philox4x64_10(uint64_t c0, uint64_t c1, uint64_t c2, uint64_t c3, uint64_t k0,
                                                    uint64_t k1) {
    const uint64_t M0 = 0xD2E7470EE14C6C93ull, M1 = 0xCA5A826395121157ull;
    const uint64_t W0 = 0x9E3779B97F4A7C15ull, W1 = 0xBB67AE8584CAA73Bull;
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        if (r > 0) { k0 += W0; k1 += W1; }
        const uint64_t hi0 = __umul64hi(M0, c0), lo0 = M0 * c0;
        const uint64_t hi1 = __umul64hi(M1, c2), lo1 = M1 * c2;
        c0 = hi1 ^ c1 ^ k0;
        c1 = lo1;
        c2 = hi0 ^ c3 ^ k1;
        c3 = lo0;
    }
    Philox4x64 out;
    out.x[0] = c0; out.x[1] = c1; out.x[2] = c2; out.x[3] = c3;
    return out;
}

// Two standard normals from two 64-bit words: ua = ((a >> 11) + 1) 2^-53 in (0, 1], ub = (b >> 11) 2^-53 in [0, 1),
// z0 = sqrt(-2 ln ua) cos(2 pi ub), z1 = sqrt(-2 ln ua) sin(2 pi ub).  ua = 1 gives (0, 0); no draw is infinite.
__device__ __forceinline__ void box_muller(uint64_t a, uint64_t b, double& z0, double& z1) {
    const double ua = (double)((a >> 11) + 1) * 0x1.0p-53;
    const double ub = (double)(b >> 11) * 0x1.0p-53;
    const double r = sqrt(-2.0 * log(ua));
    double s, c;
    sincospi(2.0 * ub, &s, &c);
    z0 = r * c;
    z1 = r * s;
}

// Four standard normals of block (counter = (run, step, stream, 0), key = (seed, 0)).
__device__ __forceinline__ void normal4(uint64_t seed, uint64_t run, uint64_t step, uint64_t stream, double z[4]) {
    const Philox4x64 p = philox4x64_10(run, step, stream, 0, seed, 0);
    box_muller(p.x[0], p.x[1], z[0], z[1]);
    box_muller(p.x[2], p.x[3], z[2], z[3]);
}

}  // namespace carmpc
