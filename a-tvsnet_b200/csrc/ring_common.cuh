// ring_common.cuh - helpers shared by the halo-ring convolution kernels (conv_ring.cu, conv_ring_s2.cu)
#pragma once
#include "tc_ptx.cuh"

namespace {

// warp-converged wait: every lane polls, the vote makes the loop condition (and everything computed
// after it) provably warp-uniform for the compiler
__device__ __forceinline__ void mbar_wait_warp(uint64_t* bar, uint32_t parity) {
    uint32_t spins = 0;
    while (!__all_sync(0xffffffffu, mbar_try_wait(bar, parity))) {
        if (++spins > TC_SPIN_LIMIT) {
            printf("atvs conv_ring: mbarrier timeout (block %d warp %d)\n", (int)blockIdx.x, (int)(threadIdx.x >> 5));
            __trap();
        }
    }
}

// MMA with the descriptors given as (lo, hi) halves: the hi halves are loop constants and the lo halves
// change by one 32-bit add per instruction
__device__ __forceinline__ void tc_mma_lohi(uint32_t tmem_d, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi,
                                            uint32_t idesc, uint32_t leader) {
    asm volatile(
        "{\n\t.reg .pred p, q;\n\t.reg .b64 ad, bd;\n\t"
        "setp.ne.b32 q, %6, 0;\n\t"
        "setp.eq.b32 p, 0, 0;\n\t"
        "mov.b64 ad, {%1, %2};\n\t"
        "mov.b64 bd, {%3, %4};\n\t"
        "@q tcgen05.mma.cta_group::1.kind::f16 [%0], ad, bd, %5, p;\n\t}" ::"r"(tmem_d),
        "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(leader)
        : "memory");
}

__device__ __forceinline__ void tc_mma_lohi1(uint32_t tmem_d, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi,
                                             uint32_t idesc) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t.reg .b64 ad, bd;\n\t"
        "setp.eq.b32 p, 0, 0;\n\t"
        "mov.b64 ad, {%1, %2};\n\t"
        "mov.b64 bd, {%3, %4};\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], ad, bd, %5, p;\n\t}" ::"r"(tmem_d),
        "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc)
        : "memory");
}

__device__ __forceinline__ void tc_ld8(uint32_t taddr, float* v) {
    uint32_t r[8];
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "r"(taddr)
                 : "memory");
#pragma unroll
    for (int i = 0; i < 8; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tc_st8_zero(uint32_t taddr) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %1, %1, %1, %1, %1, %1, %1};" ::"r"(taddr), "r"(0u)
                 : "memory");
}
__device__ __forceinline__ void tc_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// instruction descriptor WITHOUT the operand format bits (OR tc_fmt_bits(dtype) in): D = f32, M = 128, N = n
__host__ __device__ constexpr uint32_t ring_idesc(int n) {
    return (1u << 4) | ((uint32_t)(n >> 3) << 17) | ((128u >> 4) << 24);
}


// Work of one CTA of a plane-ring kernel as a sequence of units (tile column, z0, zlen): the planes of all columns form
// ONE sequence (column-major, z fastest) that is cut into gridDim.x equal ranges; a range that crosses a column end
// becomes two units.  Every CTA runs total/grid planes (+ the halo planes of its 1-2 units), whatever the volume.
// (Fixed z segments per CTA, measured before: the tile columns of a volume rarely divide by the resident CTAs - cfg2:
// 80 columns x 5 segments = 400 units on 296 CTAs = 1.35 waves, the launch lasts 2 x 28 plane steps where 37 would do.)
struct RingSpan {
    long long pos, end;
    __device__ __forceinline__ explicit RingSpan(long long total) {
        pos = total * (long long)blockIdx.x / (long long)gridDim.x;
        end = total * ((long long)blockIdx.x + 1) / (long long)gridDim.x;
    }
    // next unit: (col, z0, zlen) of the next piece of the range
    __device__ __forceinline__ bool next(int nz, long long& col, int& z0, int& zlen) {
        if (pos >= end) return false;
        col = pos / nz;
        z0 = (int)(pos - col * nz);
        zlen = (int)min((long long)(nz - z0), end - pos);
        pos += zlen;
        return true;
    }
};

// grid of a balanced launch: all resident slots, but at least `minplanes` planes per CTA.  A CTA's fixed cost (TMEM
// allocation, weight image, pipeline fill, cold first loads) is worth ~10 plane steps, and a tensor CTA holds half an
// SM's shared memory and TMEM columns while it lives.  A launch that has the GPU to itself wants many CTAs
// (`alone` planes per CTA); in a step of 8 passes on 8 streams FEWER, LONGER CTAs win (`shared` planes per CTA:
// profiles/r02_tune_step_balanced.txt on cfg2 - 5.95 ms with fixed z segments, 6.46 with 12 planes
// per CTA everywhere, 5.60 with 40 (stride 1) / 80 (stride 2) / 160 (transposed)), at the price of the launch's own
// latency (a 16-CTA transposed convolution lasts 95 us instead of 33).  The caller says how many passes it runs side
// by side (atvs_set_concurrency, 1 by default); in between the two settings are interpolated.
inline int ring_balanced_grid(long long total, long long slots, int alone, int shared) {
    long long g = slots;
    const int conc = atvs_concurrency() < 8 ? atvs_concurrency() : 8;
    const int minplanes = alone + (shared - alone) * (conc - 1) / 7;
    if (total / g < minplanes) g = total / minplanes;
    {   // small volumes: never fewer than 16 CTAs (of >= 6 planes) - a layer of 320 planes on 2 CTAs would serialise its pass
        long long floor_g = total / 6 < 16 ? total / 6 : 16;
        if (g < floor_g) g = floor_g;
    }
    if (g > total) g = total;
    if (g < 1) g = 1;
    return (int)g;
}

}  // namespace
