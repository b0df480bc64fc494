// tc_ptx.cuh - inline-PTX wrappers for the Blackwell async machinery used by the tensor-core
// convolution kernels: mbarrier, TMA (cp.async.bulk[.tensor]), tcgen05 (alloc / mma / commit /
// ld / fences), shared-memory matrix descriptors, and the shared epilogue helpers.
#pragma once
#include "common.cuh"
#include <cuda.h>

namespace {

constexpr uint32_t TC_SPIN_LIMIT = 1u << 27;   // bounded waits: trap instead of hanging the GPU

// ------------------------------------------------------------------ 16-bit operand format
// The tensor path moves its operands as opaque 16-bit words; the only places that know whether they are
// bf16 or fp16 are the instruction descriptor of tcgen05.mma.kind::f16 (A format bits [7,10), B format bits
// [10,13): 0 = f16, 1 = bf16) and the float -> 16-bit conversions of the weight packers.
__host__ __device__ constexpr uint32_t tc_fmt_bits(int dtype) { return dtype == ATVS_BF16 ? ((1u << 7) | (1u << 10)) : 0u; }
__device__ __forceinline__ unsigned short tc_cvt16(float v, int f16) {
    if (f16) return __half_as_ushort(__float2half_rn(fminf(fmaxf(v, -65504.f), 65504.f)));
    return __bfloat16_as_ushort(__float2bfloat16_rn(v));
}

// ------------------------------------------------------------------ PTX wrappers
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// suspend-time hint of mbarrier.try_wait in ns.  Measured against no hint (the hardware's default time limit,
// profiles/r02_ring_probe.txt): the kernels alone do not care, the whole cfg2 step is 0.08 ms faster with the long hint
// (waiting warps sleep instead of polling while 8 streams share the SMs).
constexpr uint32_t MBAR_HINT_NS = 10000000;
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity), "r"(MBAR_HINT_NS)
        : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    uint32_t spins = 0;
    while (!mbar_try_wait(bar, parity)) {
        if (++spins > TC_SPIN_LIMIT) {
            printf("atvs conv_tc: mbarrier timeout (block %d thread %d)\n", (int)blockIdx.x, (int)threadIdx.x);
            __trap();
        }
    }
}

__device__ __forceinline__ void tma_load_5d(void* dst, const CUtensorMap* map, int c0, int c1, int c2, int c3, int c4,
                                            uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.tensor.5d.shared::cluster.global.tile.mbarrier::complete_tx::bytes"
        " [%0], [%1, {%3, %4, %5, %6, %7}], [%2];" ::"r"(smem_u32(dst)),
        "l"((uint64_t)map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
        : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* map, int c0, int c1, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes"
        " [%0], [%1, {%3, %4}], [%2];" ::"r"(smem_u32(dst)),
        "l"((uint64_t)map), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
        : "memory");
}
// leader-predicated variants for a converged producer warp (operands stay in uniform registers)
__device__ __forceinline__ void mbar_expect_tx_leader(uint64_t* bar, uint32_t bytes, uint32_t leader) {
    asm volatile(
        "{\n\t.reg .pred q;\n\t"
        "setp.ne.b32 q, %2, 0;\n\t"
        "@q mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n\t}" ::"r"(smem_u32(bar)),
        "r"(bytes), "r"(leader)
        : "memory");
}
__device__ __forceinline__ void tma_load_5d_leader(void* dst, const CUtensorMap* map, int c0, int c1, int c2, int c3,
                                                   int c4, uint64_t* bar, uint32_t leader) {
    asm volatile(
        "{\n\t.reg .pred q;\n\t"
        "setp.ne.b32 q, %8, 0;\n\t"
        "@q cp.async.bulk.tensor.5d.shared::cluster.global.tile.mbarrier::complete_tx::bytes"
        " [%0], [%1, {%3, %4, %5, %6, %7}], [%2];\n\t}" ::"r"(smem_u32(dst)),
        "l"((uint64_t)map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4), "r"(leader)
        : "memory");
}
__device__ __forceinline__ void tma_load_2d_leader(void* dst, const CUtensorMap* map, int c0, int c1, uint64_t* bar,
                                                   uint32_t leader) {
    asm volatile(
        "{\n\t.reg .pred q;\n\t"
        "setp.ne.b32 q, %5, 0;\n\t"
        "@q cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes"
        " [%0], [%1, {%3, %4}], [%2];\n\t}" ::"r"(smem_u32(dst)),
        "l"((uint64_t)map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(leader)
        : "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* map) {
    asm volatile("prefetch.tensormap [%0];" ::"l"((uint64_t)map) : "memory");
}

__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void tc_mma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                            uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// The MMA-issuing warp runs converged (all 32 lanes execute the loop, operands are warp-uniform so
// they live in uniform registers); only the elected lane (`leader` != 0) issues the instruction.
__device__ __forceinline__ uint32_t elect_one() {
    uint32_t pred;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "elect.sync _|p, 0xffffffff;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(pred));
    return pred;
}
__device__ __forceinline__ void tc_mma_bf16_acc(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                                uint32_t leader) {
    asm volatile(
        "{\n\t.reg .pred p, q;\n\t"
        "setp.ne.b32 q, %4, 0;\n\t"
        "setp.eq.b32 p, 0, 0;\n\t"
        "@q tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(leader)
        : "memory");
}
__device__ __forceinline__ void tc_mma_bf16_first(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                                  uint32_t leader) {
    asm volatile(
        "{\n\t.reg .pred p, q;\n\t"
        "setp.ne.b32 q, %4, 0;\n\t"
        "setp.ne.b32 p, 0, 0;\n\t"
        "@q tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(leader)
        : "memory");
}
__device__ __forceinline__ void tc_commit_leader(uint64_t* bar, uint32_t leader) {
    asm volatile(
        "{\n\t.reg .pred q;\n\t"
        "setp.ne.b32 q, %1, 0;\n\t"
        "@q tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t}" ::"r"(smem_u32(bar)),
        "r"(leader)
        : "memory");
}
__device__ __forceinline__ void tc_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void tc_ld16(uint32_t taddr, float* v) {
    uint32_t r[16];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, "
        "[%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr)
        : "memory");
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tc_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// shared-memory matrix descriptor (K-major operand tile):
//   [0,14) start>>4 | [16,30) LBO>>4 | [32,46) SBO>>4 | [46,48) version=1 | [61,64) swizzle mode
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo, uint32_t sbo, uint32_t layout) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr & 0x3FFFF) >> 4);
    d |= (uint64_t)((lbo >> 4) & 0x3FFF) << 16;
    d |= (uint64_t)((sbo >> 4) & 0x3FFF) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)layout << 61;
    return d;
}

// descriptor whose start address is advanced by a byte offset (multiple of 16, no carry out of the
// 14-bit address field: shared memory is < 256 KB)
__device__ __forceinline__ uint64_t desc_advance(uint64_t d, uint32_t byte_off) { return d + (uint64_t)(byte_off >> 4); }

// 32 values per lane -> lane L ends with the sum over the warp of v[L] (31 shuffles)
__device__ __forceinline__ float warp_transpose_reduce32(float* v, int lane) {
#pragma unroll
    for (int off = 16, n = 32; off >= 1; off >>= 1, n >>= 1) {
        const bool upper = (lane & off) != 0;
#pragma unroll
        for (int i = 0; i < n / 2; ++i) {
            const float send = upper ? v[i] : v[i + n / 2];
            const float keep = upper ? v[i + n / 2] : v[i];
            v[i] = keep + __shfl_xor_sync(0xffffffffu, send, off);
        }
    }
    return v[0];
}


__device__ __forceinline__ void bulk_copy_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
        "l"((uint64_t)src), "r"(bytes), "r"(smem_u32(bar))
        : "memory");
}

// ---------------------------------------------------------------------------------------------------
// raw convolution outputs: fp32 (parity path / layers without BN) or SATURATED fp16 (layers whose output only
// feeds the batch-statistics BN pass: the moments still come from the fp32 accumulators, fp16 keeps 11
// significant bits of the value that the BN pass immediately rounds to bf16 anyway, and halves the bytes
// written here and read back there).  `off` is the ELEMENT offset of the row's first column.
//   vec: 8 = rows of 8k columns, 32-byte aligned (one STG.256 / one 16-byte fp16 store per 8 columns)
//        4 = rows of 4k columns, 16-byte aligned;  1 = scalar
__device__ __forceinline__ uint32_t pack_f16x2_sat(float lo, float hi) {
    uint32_t r;
    asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
    return r;
}
__device__ __forceinline__ int raw_vec_mode(const void* out, int ncols, int Cout, int coff) {
    if (((ncols | Cout | coff) & 7) == 0 && (((uintptr_t)out) & 31) == 0) return 8;
    if (((ncols | Cout | coff) & 3) == 0 && (((uintptr_t)out) & 15) == 0) return 4;
    return 1;
}
// `sat` (may be NULL): device counter of fp16 raw rows that held a value beyond +-65504 and were clamped
template <int NC>
__device__ __forceinline__ void store_raw_row(float* out, size_t off, const float* v, int ncols, int vec, int raw16,
                                              unsigned long long* sat = nullptr) {
    if (raw16 && sat != nullptr) {
        float m = 0.f;
#pragma unroll
        for (int c = 0; c < NC; ++c)
            if (c < ncols) m = fmaxf(m, fabsf(v[c]));
        if (m > 65504.f) atomicAdd(sat, 1ULL);
    }
    if (!raw16) {
        float* op = out + off;
        if (vec == 8) {
#pragma unroll
            for (int c = 0; c < NC; c += 8)
                if (c < ncols)
                    asm volatile("st.global.v8.f32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(op + c), "f"(v[c]),
                                 "f"(v[c + 1]), "f"(v[c + 2]), "f"(v[c + 3]), "f"(v[c + 4]), "f"(v[c + 5]), "f"(v[c + 6]),
                                 "f"(v[c + 7])
                                 : "memory");
        } else if (vec == 4) {
#pragma unroll
            for (int c = 0; c < NC; c += 4)
                if (c < ncols) *reinterpret_cast<float4*>(op + c) = make_float4(v[c], v[c + 1], v[c + 2], v[c + 3]);
        } else {
#pragma unroll
            for (int c = 0; c < NC; ++c)
                if (c < ncols) op[c] = v[c];
        }
    } else {
        __half* op = reinterpret_cast<__half*>(out) + off;
        if (vec == 8) {
#pragma unroll
            for (int c = 0; c < NC; c += 8)
                if (c < ncols) {
                    uint4 u;
                    u.x = pack_f16x2_sat(v[c], v[c + 1]); u.y = pack_f16x2_sat(v[c + 2], v[c + 3]);
                    u.z = pack_f16x2_sat(v[c + 4], v[c + 5]); u.w = pack_f16x2_sat(v[c + 6], v[c + 7]);
                    *reinterpret_cast<uint4*>(op + c) = u;
                }
        } else if (vec == 4) {
#pragma unroll
            for (int c = 0; c < NC; c += 4)
                if (c < ncols) {
                    uint2 u;
                    u.x = pack_f16x2_sat(v[c], v[c + 1]); u.y = pack_f16x2_sat(v[c + 2], v[c + 3]);
                    *reinterpret_cast<uint2*>(op + c) = u;
                }
        } else {
#pragma unroll
            for (int c = 0; c < NC; ++c)
                if (c < ncols) {
                    const uint32_t u = pack_f16x2_sat(v[c], 0.f);
                    reinterpret_cast<unsigned short*>(op)[c] = (unsigned short)(u & 0xffffu);
                }
        }
    }
}

// epilogue of one 128-row accumulator tile: TMEM -> registers, raw fp32 store of the real columns,
// per-channel sum / sum of squares folded into per-lane running registers (batch-stat BN).
template <int NPAD>
__device__ __forceinline__ void epilogue_tile(uint32_t taddr, uint64_t* tempty_bar, int lane, bool valid, float* out,
                                              size_t off, int ncols, int vec, int raw16, bool want_stats, float* run,
                                              const float* bias_row = nullptr, unsigned long long* sat = nullptr,
                                              bool relu = false) {
    const bool vec4 = vec >= 4;
    float v[NPAD];
#pragma unroll
    for (int c = 0; c < NPAD; c += 16) tc_ld16(taddr + c, v + c);
    tc_wait_ld();
    tc_fence_before();
    __syncwarp();
    if (lane == 0 && tempty_bar != nullptr) mbar_arrive(tempty_bar);
    if (bias_row != nullptr && valid) {
        // depth-invariant part of the layer (the tiled reference-feature half of the cost volume)
        if (vec4) {
#pragma unroll
            for (int c = 0; c < NPAD; c += 4)
                if (c < ncols) {
                    const float4 bv = __ldg(reinterpret_cast<const float4*>(bias_row + c));
                    v[c] += bv.x; v[c + 1] += bv.y; v[c + 2] += bv.z; v[c + 3] += bv.w;
                }
        } else {
#pragma unroll
            for (int c = 0; c < NPAD; ++c)
                if (c < ncols) v[c] += __ldg(bias_row + c);
        }
    }
    if (relu) {
#pragma unroll
        for (int c = 0; c < NPAD; ++c) v[c] = fmaxf(v[c], 0.f);
    }
    if (valid) store_raw_row<NPAD>(out, off, v, ncols, vec, raw16, sat);
    if (want_stats && valid) {
        // per-THREAD running moments (row = this thread's voxel): no cross-lane traffic per tile
#pragma unroll
        for (int c = 0; c < NPAD; ++c) {
            run[c] += v[c];
            run[NPAD + c] = fmaf(v[c], v[c], run[NPAD + c]);
        }
    }
}

// flush the per-thread running statistics (run[0..NPAD) sums, run[NPAD..2NPAD) sums of squares):
// one transposed warp reduction per 32 values, then stats[c] += sum, stats[Cout + c] += sum of squares
template <int NPAD>
__device__ __forceinline__ void flush_stats(double* stats, float* run, int lane, int Cout, int coff, int ncols) {
#pragma unroll
    for (int h = 0; h < (2 * NPAD) / 32; ++h) {
        const float tot = warp_transpose_reduce32(run + h * 32, lane);
        const int idx = h * 32 + lane;                 // index into [sums | sums of squares]
        const int c = idx % NPAD;
        if (c < ncols) atomicAdd(&stats[(idx < NPAD ? 0 : Cout) + coff + c], (double)tot);
    }
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

inline EncodeTiledFn get_encode() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
            qres == cudaDriverEntryPointSuccess)
            fn = (EncodeTiledFn)p;
    }
    return fn;
}

}  // namespace
