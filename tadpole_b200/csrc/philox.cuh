// philox.cuh -- Philox4x32-10 (Salmon, Moraes, Dror, Shaw 2011), the counter-based generator of every random draw the
// library makes: diffT's random partitions (difft.cu, counter word 3 = 0x7ad) and the equal-depth subsamples
// (downsample.cu, counter word 3 = 0xD5000000 | chromosome).  A draw is a function of (counter, seed) alone, so a kernel
// regenerates any key whenever it needs it instead of storing it.  oracle/tadpole_oracle.py restates it (philox4x32).
#pragma once

// the first 64 bits (x0 << 32 | x1) of Philox4x32-10 on counter (c0, c1, c2, c3) with key = (seed low, seed high)
__host__ __device__ __forceinline__ unsigned long long philox4x32_key64(unsigned c0, unsigned c1, unsigned c2, unsigned c3,
                                                                        unsigned long long seed) {
    unsigned k0 = (unsigned)seed, k1 = (unsigned)(seed >> 32);
    unsigned x0 = c0, x1 = c1, x2 = c2, x3 = c3;
#pragma unroll
    for (int r = 0; r < 10; r++) {
        const unsigned long long p0 = (unsigned long long)0xD2511F53u * x0, p1 = (unsigned long long)0xCD9E8D57u * x2;
        const unsigned y0 = (unsigned)(p1 >> 32) ^ x1 ^ k0, y1 = (unsigned)p1;
        const unsigned y2 = (unsigned)(p0 >> 32) ^ x3 ^ k1, y3 = (unsigned)p0;
        x0 = y0; x1 = y1; x2 = y2; x3 = y3;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    return ((unsigned long long)x0 << 32) | x1;
}
