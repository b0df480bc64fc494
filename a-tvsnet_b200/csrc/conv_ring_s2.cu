// conv_ring_s2.cu - stride-2 3x3x3 convolution (network.py:173-215 conv_bn, strides=2; TF 'SAME' on even
// extents = padding (0,1), SURVEY.md Appendix C) as a tcgen05 implicit GEMM over a shared-memory ring
// of input planes, for the large volumes (conv_b*_1_0: full resolution -> 1/8 of the voxels).
//
// Same pipeline as conv_ring.cu (4 producer warps | one MMA-issuing thread | 4 epilogue warps, every
// input plane consumed once, the z taps side by side in the MMA N dimension), with two differences:
//   * an output row of the MMA tile reads every OTHER input voxel, but the rows of a no-swizzle core
//     matrix must be 16 bytes apart: the producers therefore DE-INTERLEAVE the halo plane into its
//     four (y parity, x parity) sub-planes while staging it, and tap (dy,dx) reads sub-plane
//     (dy&1, dx&1) at the offset (dy>>1, dx>>1);
//   * out[k] = sum_dz in[2k+dz] w[dz]: an even input plane 2j feeds the output planes j-1 (dz=2) and
//     j (dz=0) in one MMA of N = 2*CP, an odd plane 2j+1 feeds plane j (dz=1) with N = CP.
//
//   work unit : one 16(y) x 8(x) output tile over an output z segment [z0, z0+zlen)
//   ring slot : [Cin/8 chunks][4 sub-planes][17 x 9 voxels][8 channels] bf16 of one input plane
//   weights   : per K=16 step [2 chunks][w_dz2 | w_dz0 | w_dz1][8 channels]
#include "ring_common.cuh"
#include "conv_ring.cuh"
#include <cstring>

namespace {

constexpr int S2_TY = 16, S2_TX = 8;
constexpr int S2_IH = 2 * S2_TY + 1, S2_IW = 2 * S2_TX + 1;      // input region of a tile: 33 x 17
constexpr int S2_SR = S2_TY + 1, S2_SC = S2_TX + 1;               // sub-plane extent: 17 x 9
constexpr int S2_SUB = S2_SR * S2_SC;                             // 153 voxel slots per sub-plane
constexpr int S2_PITCH = 4 * S2_SUB * 16 + 16;                    // one 8-channel chunk of a plane (+16: banks)
constexpr int S2_PRODUCERS = 128;
constexpr int S2_THREADS = 288;
constexpr int S2_G = 8;                                           // accumulator groups (output planes) in TMEM

struct S2Params {
    int B, D, H, W;             // input extents
    int Do, Ho, Wo;
    int Cout, coff, ncols;
    int raw16;                  // raw output dtype: 0 fp32, 1 saturated fp16
    uint32_t fmt;               // operand format bits of the instruction descriptor (tc_fmt_bits)
    unsigned long long* sat;    // saturation counter of the fp16 raw stores (atvs_sat_ptr)
    int nXT, nYT;
    int nring;
    int wbytes;
    long long total;            // tile columns * Do: the output plane sequence cut into one range per CTA (RingSpan)
};

template <int CIN, int CP>
struct S2Cfg {
    static constexpr int NKC = CIN / 8;                             // 8-channel chunks per slot
    static constexpr int SLOT_BYTES = (NKC * S2_PITCH + 127) / 128 * 128;
    static constexpr int NSTEPS = (CIN >= 16) ? 9 * (CIN / 16) : 5;
    static constexpr int NROWS = 3 * CP;
    static constexpr int STEP_BYTES = 2 * NROWS * 16;
    static constexpr uint32_t TMEM_COLS = (uint32_t)(S2_G * CP);   // 128 or 256
};

struct S2Unit {
    int b, x0, y0, z0, zlen;
};

struct S2Iter {
    RingSpan span;
    __device__ __forceinline__ explicit S2Iter(const S2Params& p) : span(p.total) {}
    __device__ __forceinline__ bool next(const S2Params& p, S2Unit& r) {
        long long t;
        if (!span.next(p.Do, t, r.z0, r.zlen)) return false;
        r.x0 = (int)(t % p.nXT) * S2_TX;
        t /= p.nXT;
        r.y0 = (int)(t % p.nYT) * S2_TY;
        r.b = (int)(t / p.nYT);
        return true;
    }
};
// input planes of a unit: i in [0, iend], plane i = input plane 2*z0 + i; the plane behind the volume
// ('SAME' padding) is skipped
__device__ __forceinline__ int s2_iend(const S2Params& p, const S2Unit& u) {
    return (2 * (u.z0 + u.zlen) < p.D) ? 2 * u.zlen : 2 * u.zlen - 1;
}

// shared-memory offset (bytes, inside one chunk) of in-plane tap (dy, dx) for the tile's first row
__host__ __device__ constexpr uint32_t s2_tap_off(int tap) {
    return (uint32_t)((((((tap / 3) & 1) << 1) | ((tap % 3) & 1)) * S2_SUB + ((tap / 3) >> 1) * S2_SC + ((tap % 3) >> 1)) * 16);
}
// Cin = 8: tap pairs of one K=16 step, ordered so that the second tap lies behind the first in shared
// memory (LBO is unsigned); the 9th tap is paired with a zero-weighted re-read of tap 7
__host__ __device__ constexpr int s2_pair_a(int s) { return s == 0 ? 0 : s == 1 ? 2 : s == 2 ? 5 : s == 3 ? 6 : 8; }
__host__ __device__ constexpr int s2_pair_b(int s) { return s == 0 ? 1 : s == 1 ? 3 : s == 2 ? 4 : s == 3 ? 7 : 7; }

template <int CIN, int CP, int MINB>
__global__ void __launch_bounds__(S2_THREADS, MINB)
k_conv3d_ring_s2(const uint16_t* __restrict__ x, const __grid_constant__ S2Params p,
                 const uint8_t* __restrict__ wimg, float* __restrict__ out, double* __restrict__ stats,
                 const float* __restrict__ bias) {
    using Cfg = S2Cfg<CIN, CP>;
    constexpr int G = S2_G;

    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>(((uintptr_t)smem_raw + 127) & ~(uintptr_t)127);
    uint8_t* wsm = smem;
    uint8_t* ring = smem + ((p.wbytes + 127) & ~127);
    uint64_t* bars = reinterpret_cast<uint64_t*>(ring + (size_t)p.nring * Cfg::SLOT_BYTES);
    uint64_t* full = bars;
    uint64_t* empty = bars + p.nring;
    uint64_t* tfull = bars + 2 * p.nring;
    uint64_t* tempty = tfull + G;
    uint64_t* wbar = tempty + G;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(wbar + 1);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int R = p.nring;
    if (threadIdx.x == 0) {
        for (int s = 0; s < R; ++s) {
            mbar_init(&full[s], S2_PRODUCERS / 32);      // one arrival per producer WARP (lane 0, after __syncwarp)
            mbar_init(&empty[s], 1);
        }
        for (int g = 0; g < G; ++g) {
            mbar_init(&tfull[g], 1);
            mbar_init(&tempty[g], 4);
        }
        mbar_init(wbar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 4) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                     "r"(Cfg::TMEM_COLS)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    if (warp >= 5) {
        // accumulation is always "+=": start from zero accumulators
        const uint32_t taddr = tmem_base + ((uint32_t)((warp & 3) * 32) << 16);
        for (uint32_t c = 0; c < Cfg::TMEM_COLS; c += 8) tc_st8_zero(taddr + c);
        tc_wait_st();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();

    if (warp < 4) {
        // ===================== producers: global -> de-interleaved ring planes =====================
        const int ptid = threadIdx.x;
        if (ptid == 0) {
            mbar_expect_tx(wbar, (uint32_t)p.wbytes);
            bulk_copy_g2s(wsm, wimg, (uint32_t)p.wbytes, wbar);
        }
        constexpr int NVOX = S2_IH * S2_IW;                         // 561 input voxels per plane and tile
        constexpr int NITEM = (Cfg::NKC * NVOX + S2_PRODUCERS - 1) / S2_PRODUCERS;
        const int PF = (R >= 5) ? 4 : (R >= 3 ? 2 : 1);
        uint32_t slot = 0, sphase = 0, pslot = 0, pending = 0;
        const uint32_t ring_u32 = smem_u32(ring);
        auto publish = [&](int keep) {
            if (keep >= 3) asm volatile("cp.async.wait_group 3;" ::: "memory");
            else if (keep == 2) asm volatile("cp.async.wait_group 2;" ::: "memory");
            else if (keep == 1) asm volatile("cp.async.wait_group 1;" ::: "memory");
            else asm volatile("cp.async.wait_group 0;" ::: "memory");
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            // every lane's copies have landed and are visible to the async proxy; one release-arrive per warp
            // (128 per-thread arrivals on one mbarrier cost more than the plane's cp.async issue)
            __syncwarp();
            for (; pending > (uint32_t)keep; --pending) {
                if ((threadIdx.x & 31) == 0) mbar_arrive(&full[pslot]);
                if (++pslot == (uint32_t)R) pslot = 0;
            }
        };
        const size_t zstride_in = (size_t)p.H * p.W * CIN;
        S2Iter units(p);
        S2Unit un;
        while (units.next(p, un)) {
            const int iend = s2_iend(p, un);
            int goff[NITEM];       // element offset inside an input z plane, -1 = zero fill, -2 = no item
#pragma unroll
            for (int k = 0; k < NITEM; ++k) {
                const int j = ptid + k * S2_PRODUCERS;
                const int c = j % Cfg::NKC, v = j / Cfg::NKC;
                const int iy = v / S2_IW, ix = v - iy * S2_IW;
                const int gy = 2 * un.y0 + iy, gx = 2 * un.x0 + ix;
                const bool ok = gy < p.H && gx < p.W;
                goff[k] = (j >= Cfg::NKC * NVOX) ? -2 : (ok ? (gy * p.W + gx) * CIN + c * 8 : -1);
            }
            const uint16_t* zbase = x + ((size_t)un.b * p.D + 2 * un.z0) * zstride_in;
            for (int i = 0; i <= iend; ++i, zbase += zstride_in) {
                mbar_wait(&empty[slot], sphase ^ 1);
                const uint32_t dst0 = ring_u32 + slot * (uint32_t)Cfg::SLOT_BYTES;
#pragma unroll
                for (int k = 0; k < NITEM; ++k) {
                    if (goff[k] != -2) {
                        const int j = ptid + k * S2_PRODUCERS;
                        const int c = j % Cfg::NKC, v = j / Cfg::NKC;
                        const int iy = v / S2_IW, ix = v - iy * S2_IW;
                        const uint32_t soff = (uint32_t)(c * S2_PITCH +
                                                         ((((iy & 1) << 1) | (ix & 1)) * S2_SUB + (iy >> 1) * S2_SC + (ix >> 1)) * 16);
                        const bool ok = goff[k] >= 0;
                        const uint16_t* src = ok ? zbase + goff[k] : x;
                        asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst0 + soff), "l"(src),
                                     "r"(ok ? 16 : 0)
                                     : "memory");
                    }
                }
                asm volatile("cp.async.commit_group;" ::: "memory");
                if (++slot == (uint32_t)R) { slot = 0; sphase ^= 1; }
                if (++pending >= (uint32_t)PF) publish(PF - 1);
            }
        }
        publish(0);
    } else if (warp == 4) {
        // ===================== MMA issuer (one elected thread, uniform datapath) =====================
        if (elect_one()) {
            mbar_wait(wbar, 0);
            tc_fence_after();
            constexpr uint32_t A_HI = (uint32_t)((S2_SC * 16) >> 4) | (1u << 14);          // SBO = next output row
            constexpr uint32_t B_HI = (uint32_t)(128 >> 4) | (1u << 14);
            constexpr uint32_t A_LBO = (CIN >= 16) ? ((uint32_t)(S2_PITCH >> 4) << 16) : 0u;
            const uint32_t a_lo_ring = (smem_u32(ring) >> 4) | A_LBO;
            const uint32_t b_lo0 = (smem_u32(wsm) >> 4) | ((uint32_t)((Cfg::NROWS * 16) >> 4) << 16);
            auto issue_plane = [&](uint32_t dcol, uint32_t a_lo0, uint32_t b_lo, uint32_t idesc) {
                constexpr int KS = (CIN >= 16) ? CIN / 16 : 1;
#pragma unroll
                for (int s = 0; s < Cfg::NSTEPS; ++s) {
                    uint32_t aoff;
                    if (CIN >= 16) {
                        const int tp = s / KS, ks = s % KS;
                        aoff = (uint32_t)((2 * ks * S2_PITCH) >> 4) + (s2_tap_off(tp) >> 4);
                    } else {
                        const uint32_t offa = s2_tap_off(s2_pair_a(s)), offb = s2_tap_off(s2_pair_b(s));
                        aoff = (offa >> 4) | (((offb - offa) >> 4) << 16);
                    }
                    tc_mma_lohi1(dcol, a_lo0 + aoff, A_HI, b_lo + ((uint32_t)(s * Cfg::STEP_BYTES) >> 4), B_HI, idesc);
                }
            };
            // weight windows (rows): [w2 | w0 | w1]
            constexpr uint32_t W_W2W0 = 0u, W_W0 = (uint32_t)CP, W_W1 = 2u * (uint32_t)CP;
            uint32_t slot = 0, sphase = 0;
            uint32_t gq = 0, gphase = 0;       // accumulator group / phase of output plane t = 0 of the unit
            S2Iter units(p);
            S2Unit un;
            while (units.next(p, un)) {
                const int iend = s2_iend(p, un);
                uint32_t gw = gq, gwphase = gphase;    // next output plane to wait for (fresh accumulator)
                uint32_t gcur = gq;                    // group of output plane j = i >> 1
                uint32_t gdone = gq;
                int tdone = 0;
                for (int i = 0; i <= iend; ++i) {
                    const int j = i >> 1;
                    const bool even = (i & 1) == 0;
                    if (even && j < un.zlen) {         // first touch of output plane j
                        mbar_wait(&tempty[gw], gwphase ^ 1);
                        if (++gw == (uint32_t)G) { gw = 0; gwphase ^= 1; }
                    }
                    const uint32_t gprev = (gcur == 0) ? (uint32_t)G - 1 : gcur - 1;
                    mbar_wait(&full[slot], sphase);
                    tc_fence_after();
                    const uint32_t a_lo0 = a_lo_ring + slot * (uint32_t)(Cfg::SLOT_BYTES >> 4);
                    if (!even) {
                        issue_plane(tmem_base + gcur * (uint32_t)CP, a_lo0, b_lo0 + ((W_W1 * 16u) >> 4), ring_idesc(CP) | p.fmt);
                    } else if (j == 0) {
                        issue_plane(tmem_base + gcur * (uint32_t)CP, a_lo0, b_lo0 + ((W_W0 * 16u) >> 4), ring_idesc(CP) | p.fmt);
                    } else if (j >= un.zlen) {
                        issue_plane(tmem_base + gprev * (uint32_t)CP, a_lo0, b_lo0 + ((W_W2W0 * 16u) >> 4), ring_idesc(CP) | p.fmt);
                    } else if (gcur != 0) {
                        issue_plane(tmem_base + gprev * (uint32_t)CP, a_lo0, b_lo0 + ((W_W2W0 * 16u) >> 4), ring_idesc(2 * CP) | p.fmt);
                    } else {                           // the pair wraps around the accumulator ring
                        issue_plane(tmem_base + gprev * (uint32_t)CP, a_lo0, b_lo0 + ((W_W2W0 * 16u) >> 4), ring_idesc(CP) | p.fmt);
                        issue_plane(tmem_base, a_lo0, b_lo0 + ((W_W0 * 16u) >> 4), ring_idesc(CP) | p.fmt);
                    }
                    tc_commit(&empty[slot]);
                    if (++slot == (uint32_t)R) { slot = 0; sphase ^= 1; }
                    // output planes whose last contribution this was
                    const int tlast = (i == iend) ? un.zlen - 1 : (even ? j - 1 : -1);
                    while (tdone <= tlast) {
                        tc_commit(&tfull[gdone]);
                        ++tdone;
                        if (++gdone == (uint32_t)G) gdone = 0;
                    }
                    if (!even && ++gcur == (uint32_t)G) gcur = 0;
                }
                gq = gw; gphase = gwphase;
            }
        }
        __syncwarp();
    } else {
        // ===================== epilogue (4 warps = 128 TMEM lanes) =====================
        const int g = warp & 3;
        const int row = g * 32 + lane;
        const int ty = row >> 3, tx = row & 7;
        float run[2 * CP];
#pragma unroll
        for (int k = 0; k < 2 * CP; ++k) run[k] = 0.f;
        const bool vec4 = (p.ncols & 3) == 0 && (p.Cout & 3) == 0;
        const int vec = raw_vec_mode(out, p.ncols, p.Cout, p.coff);
        uint32_t grp = 0, gphase = 0;
        S2Iter units(p);
        S2Unit un;
        while (units.next(p, un)) {
            const int y = un.y0 + ty, xq = un.x0 + tx;
            const bool valid = y < p.Ho && xq < p.Wo;
            const size_t obase = valid ? ((((size_t)un.b * p.Do + un.z0) * p.Ho + y) * p.Wo + xq) * p.Cout + p.coff : 0;
            const size_t zstride = (size_t)p.Ho * p.Wo * p.Cout;
            for (int t = 0; t < un.zlen; ++t) {
                mbar_wait(&tfull[grp], gphase);
                tc_fence_after();
                const uint32_t taddr = tmem_base + ((uint32_t)(g * 32) << 16) + grp * (uint32_t)CP;
                uint64_t* const tempty_bar = &tempty[grp];
                if (++grp == (uint32_t)G) { grp = 0; gphase ^= 1; }
                float v[CP];
#pragma unroll
                for (int c = 0; c < CP; c += 8) tc_ld8(taddr + c, v + c);
                tc_wait_ld();
#pragma unroll
                for (int c = 0; c < CP; c += 8) tc_st8_zero(taddr + c);
                tc_wait_st();
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(tempty_bar);
                if (!valid) continue;
                const size_t ooff = obase + (size_t)t * zstride;
                if (bias != nullptr) {
                    // depth-invariant part of the layer (the tiled reference-feature half of the cost volume)
                    const int z = un.z0 + t;
                    const int zc = (z == 0) ? 0 : (z == p.Do - 1 ? 2 : 1);
                    const float* brow = bias + ((((size_t)un.b * 3 + zc) * p.Ho + y) * p.Wo + xq) * p.Cout + p.coff;
                    if (vec4) {
#pragma unroll
                        for (int c = 0; c < CP; c += 4)
                            if (c < p.ncols) {
                                const float4 bv = __ldg(reinterpret_cast<const float4*>(brow + c));
                                v[c] += bv.x; v[c + 1] += bv.y; v[c + 2] += bv.z; v[c + 3] += bv.w;
                            }
                    } else {
#pragma unroll
                        for (int c = 0; c < CP; ++c)
                            if (c < p.ncols) v[c] += __ldg(brow + c);
                    }
                }
                store_raw_row<CP>(out, ooff, v, p.ncols, vec, p.raw16, p.sat);
                if (stats != nullptr) {
#pragma unroll
                    for (int c = 0; c < CP; ++c) {
                        run[c] += v[c];
                        run[CP + c] = fmaf(v[c], v[c], run[CP + c]);
                    }
                }
            }
        }
        if (stats != nullptr) {
#pragma unroll
            for (int k = 0; k < 2 * CP; ++k) {
                float tot = run[k];
#pragma unroll
                for (int off = 16; off >= 1; off >>= 1) tot += __shfl_xor_sync(0xffffffffu, tot, off);
                const int c = k % CP;
                if (lane == 0 && c < p.ncols) atomicAdd(&stats[(k < CP ? 0 : p.Cout) + p.coff + c], (double)tot);
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 4) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(Cfg::TMEM_COLS)
                     : "memory");
    }
}

// weight image of one Cout slab: [step][2 chunks][w_dz2 | w_dz0 | w_dz1 rows of CP][8 channels] bf16
__global__ void k_pack_ring_s2(const float* __restrict__ w, int Cin, int Cout, int cp, int f16, unsigned short* __restrict__ out) {
    const int nsteps = ring_nsteps(Cin);
    const int nrows = 3 * cp;
    const int slab = blockIdx.x / nsteps, step = blockIdx.x % nsteps;
    unsigned short* o = out + ((size_t)slab * nsteps + step) * 2 * nrows * 8;
    for (int i = threadIdx.x; i < 2 * nrows * 8; i += blockDim.x) {
        const int chunk = i / (nrows * 8), r = (i / 8) % nrows, e = i % 8;
        const int grp = r / cp, n = r % cp;
        const int dz = grp == 0 ? 2 : (grp == 1 ? 0 : 1);
        int tap2d, k;
        if (Cin >= 16) {
            tap2d = step / (Cin / 16);
            k = ((step % (Cin / 16)) * 2 + chunk) * 8 + e;
        } else {
            tap2d = chunk == 0 ? s2_pair_a(step) : (step == 4 ? -1 : s2_pair_b(step));
            k = e;
        }
        const int co = slab * cp + n;
        float val = 0.f;
        if (tap2d >= 0 && co < Cout) val = w[((size_t)(dz * 9 + tap2d) * Cin + k) * Cout + co];
        o[i] = tc_cvt16(val, f16);
    }
}

template <int CIN, int CP, int MINB>
int launch_s2(const uint16_t* x, const S2Params& p, const uint8_t* wimg, float* out, double* stats,
              const float* bias, size_t smem, int grid, cudaStream_t st) {
    if (const int rc = atvs_max_dynamic_smem<k_conv3d_ring_s2<CIN, CP, MINB>>()) return rc;
    k_conv3d_ring_s2<CIN, CP, MINB><<<grid, S2_THREADS, smem, st>>>(x, p, wimg, out, stats, bias);
    ATVS_LAUNCH_CHECK();
    return 0;
}

int s2_cp(int Cout) { return Cout <= 16 ? 16 : 32; }
size_t s2_slab_bytes(int Cin, int cp) { return (size_t)ring_nsteps(Cin) * 2 * 3 * cp * 16; }

}  // namespace

// Cin = 32 needs ~200 KB of ring planes per CTA (or two K phases of 16 channels per plane to fit two CTAs per SM):
// standalone it beats the per-tap TMA kernel (73 vs 88 us at cfg2), but it monopolises the SM while the other streams
// of a step want to co-run (measured +0.25 ms per depth map), so the 32-channel layers stay on the per-tap kernel
bool ring_s2_supported(int Cin, int Cout) { return (Cin == 8 || Cin == 16) && Cout >= 1 && Cout <= 64; }

size_t ring_s2_weight_bytes(int Cin, int Cout) {
    if (!ring_s2_supported(Cin, Cout)) return 0;
    const int cp = s2_cp(Cout);
    return (size_t)((Cout + cp - 1) / cp) * s2_slab_bytes(Cin, cp);
}

int ring_s2_pack(const float* kernel, int Cin, int Cout, int dtype, void* wimg, cudaStream_t st) {
    const int cp = s2_cp(Cout);
    const int nslabs = (Cout + cp - 1) / cp;
    k_pack_ring_s2<<<nslabs * ring_nsteps(Cin), 128, 0, st>>>(kernel, Cin, Cout, cp, dtype == ATVS_F16, (unsigned short*)wimg);
    ATVS_LAUNCH_CHECK();
    return 0;
}

// output voxels from which the plane ring replaces the per-tap TMA kernel (131072 -> 32768: 5.03 -> 5.00 ms per cfg2
// depth map)
constexpr long long RING_S2_MINVOX = 32768;
bool ring_s2_applicable(int B, int D, int H, int W, int Cin, int Cout) {
    return ring_s2_supported(Cin, Cout) && ((D | H | W) & 1) == 0 && (long long)(D / 2) * (H / 2) * (W / 2) >= RING_S2_MINVOX;
}

int ring_s2_conv(const void* x16, int dtype, const void* wimg, int B, int D, int H, int W, int Cin, int Cout, float* raw_out,
                 int raw16, double* stats, const float* bias, cudaStream_t st) {
    const int cp = s2_cp(Cout);
    const int nslabs = (Cout + cp - 1) / cp;
    const int sms = atvs_num_sms();
    S2Params p;
    memset(&p, 0, sizeof(p));
    p.B = B; p.D = D; p.H = H; p.W = W; p.Do = D / 2; p.Ho = H / 2; p.Wo = W / 2; p.Cout = Cout;
    p.raw16 = raw16;
    p.fmt = tc_fmt_bits(dtype);
    p.sat = raw16 ? atvs_sat_ptr() : nullptr;
    p.nXT = (p.Wo + S2_TX - 1) / S2_TX;
    p.nYT = (p.Ho + S2_TY - 1) / S2_TY;
    p.wbytes = (int)s2_slab_bytes(Cin, cp);
    const size_t slot = ((size_t)(Cin / 8) * S2_PITCH + 127) / 128 * 128;
    const size_t fixed = 128 + (size_t)((p.wbytes + 127) & ~127) + (2 * 8 + 2 * S2_G + 1) * 8 + 16;
    const int minb = (cp < 32 && fixed + 4 * slot <= 110 * 1024) ? 2 : 1;
    const size_t budget = (minb == 2 ? 110 : 220) * 1024;
    int nring = (int)((budget - fixed) / slot);
    if (nring > 8) nring = 8;
    if (nring < 2) {
        atvs_set_error("atvs_conv3d_bf16(ring s2): weights do not fit next to 2 ring planes (Cin=%d Cout=%d)", Cin, Cout);
        return ATVS_E_UNSUP;
    }
    p.nring = nring;
    p.total = (long long)B * p.nXT * p.nYT * p.Do;
    const size_t smem = fixed + (size_t)nring * slot;
    const int grid = ring_balanced_grid(p.total, (long long)sms * minb, 20, 80);
    for (int slab = 0; slab < nslabs; ++slab) {
        p.coff = slab * cp;
        p.ncols = (Cout - p.coff < cp) ? Cout - p.coff : cp;
        const uint8_t* wi = (const uint8_t*)wimg + (size_t)slab * p.wbytes;
        int rc = 0;
#define S2_CASE(CI, CPV)                                                                                             \
    if (Cin == CI && cp == CPV) {                                                                                    \
        rc = (minb == 2) ? launch_s2<CI, CPV, 2>((const uint16_t*)x16, p, wi, raw_out, stats, bias, smem, grid, st) \
                         : launch_s2<CI, CPV, 1>((const uint16_t*)x16, p, wi, raw_out, stats, bias, smem, grid, st); \
    } else
        S2_CASE(8, 16) S2_CASE(8, 32) S2_CASE(16, 16) S2_CASE(16, 32)
        {
            atvs_set_error("atvs_conv3d_bf16(ring s2): no kernel for Cin=%d CP=%d", Cin, cp);
            return ATVS_E_UNSUP;
        }
#undef S2_CASE
        if (rc) return rc;
    }
    return 0;
}
