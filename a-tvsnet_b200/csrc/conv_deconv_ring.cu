// conv_deconv_ring.cu - stride-2 transposed 3x3x3 convolution (network.py:511-550 deconv_bn,
// tf.layers.conv3d_transpose 'SAME': out[2i+k] += in[i]*w[k], cropped to [0, 2n)) as a tcgen05 implicit GEMM
// over a shared-memory RING OF INPUT PLANES, sub-pixel form.
//
// Per dimension an output pair (2j, 2j+1) reads in[j] (k = 0 -> 2j, k = 1 -> 2j+1) and in[j-1] (k = 2 -> 2j), so
//   * in the plane, an M = 128 tile of 16 x 8 pair positions needs the input tile at the four shifts (0|-1, 0|-1):
//     the ring slot holds the tile with a one-voxel halo on the LOW side (17 x 9) and the shifts are UMMA
//     descriptor offsets into it (no-swizzle K-major core matrices, as conv_ring.cu);
//   * along z, input plane z feeds the output planes 2z (kz=0), 2z+1 (kz=1) and 2z+2 (kz=2).
// The N dimension of one MMA carries [3 output planes][4 in-plane parity classes][Cout]: an accumulator group
// (4*Cout TMEM columns) per OUTPUT plane in a ring of 8 groups, and per input plane 4 shifts x Cin/16 MMAs with
// N = 12*Cout over three consecutive groups (weights of (class, shift) pairs that have no tap are zero).  That is
// 4 MMAs (N = 96) per 128 input voxels for 16 -> 8 instead of the 27 (N = 16) of the per-(class, tap) kernel
// (conv_deconv.cu), and every input voxel is staged ONCE (plus halo) instead of 8 shifted TMA tiles: the kernel is
// bound by the write of its 8x larger output.
//
//   work unit : a 16(y) x 8(x) tile of input positions over an input z segment [z0, z0+zlen) (+ plane z0-1,
//               whose kz=2 taps complete output plane 2*z0)
//   warps 0-3 producers (cp.async, zero fill = outside the volume) | warp 4 MMA issuer | warps 5-12 epilogue:
//   two sets of four warps (one per TMEM lane quarter), set 0 drains the even output planes, set 1 the odd ones -
//   the per-role timelines (profiles/r02_deconv_ring_trace.txt) showed ONE set as the critical
//   path at ~1600 cycles per input plane (convert + store + moments of 2 x 128 x 32 values on 4 warps) with the MMA
//   warp waiting for accumulators.  Accumulation is always "+=": the epilogue zeroes a group right after reading it.
#include "ring_common.cuh"
#include "conv_deconv.cuh"
#include <cstring>

namespace {

constexpr int DR_TY = 16, DR_TX = 8, DR_HH = DR_TY + 1, DR_WW = DR_TX + 1;
constexpr int DR_NVOX = DR_HH * DR_WW;              // voxels of one halo plane (153)
constexpr int DR_KCH_PAD = DR_NVOX * 16 + 16;       // pitch of one 8-channel chunk plane (+16 B: bank skew)
constexpr int DR_PRODUCERS = 128;
constexpr int DR_THREADS = 416;                     // 4 producer + 1 MMA + 8 epilogue warps
constexpr int DR_G = 8;                              // accumulator groups (output planes) in TMEM
constexpr int DR_MAXR = 16;                          // ring slots (mbarrier pairs)

struct DrParams {
    int B, D, H, W;         // INPUT extents
    int Cout;
    int raw16;              // raw output dtype: 0 fp32, 1 saturated fp16
    uint32_t fmt;           // operand format bits of the instruction descriptor (tc_fmt_bits)
    unsigned long long* sat;   // saturation counter of the fp16 raw stores (atvs_sat_ptr)
    int nXT, nYT;
    int nring, pf;
    int wbytes;
    long long total;        // tile columns * D: the input plane sequence cut into one range per CTA (RingSpan)
};

template <int CIN, int COUT>
struct DrCfg {
    static constexpr int NKC = CIN / 8;
    static constexpr int SLOT_BYTES = (NKC * DR_KCH_PAD + 127) / 128 * 128;
    static constexpr int KS = CIN / 16;
    static constexpr int NSTEPS = 4 * KS;                 // (shift, K=16 step) MMAs per input plane
    static constexpr int GC = 4 * COUT;                   // columns of one output plane: [class][co]
    static constexpr int NROWS = 3 * GC;                  // rows of one weight step image: [kz0 | kz1 | kz2]
    static constexpr int STEP_BYTES = 2 * NROWS * 16;
    static constexpr uint32_t TMEM_COLS = (uint32_t)(DR_G * GC);    // 256 (Cout 8) or 512 (Cout 16)
};

struct DrUnit {
    int b, x0, y0, z0, zlen;
};


struct DrIter {
    RingSpan span;
    __device__ __forceinline__ explicit DrIter(const DrParams& p) : span(p.total) {}
    __device__ __forceinline__ bool next(const DrParams& p, DrUnit& r) {
        long long t;
        if (!span.next(p.D, t, r.z0, r.zlen)) return false;
        r.x0 = (int)(t % p.nXT) * DR_TX;
        t /= p.nXT;
        r.y0 = (int)(t % p.nYT) * DR_TY;
        r.b = (int)(t / p.nYT);
        return true;
    }
};

// 16 consecutive fp32 values -> 16 saturated halves, ONE 32-byte store (p 32-byte aligned)
__device__ __forceinline__ void store_f16x16(__half* p, const float* v) {
    uint32_t r[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) r[i] = pack_f16x2_sat(v[2 * i], v[2 * i + 1]);
    asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(p), "r"(r[0]), "r"(r[1]), "r"(r[2]),
                 "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
                 : "memory");
}

template <int CIN, int COUT>
__global__ void __launch_bounds__(DR_THREADS, 1)
k_deconv3d_ring(const uint16_t* __restrict__ x, const __grid_constant__ DrParams p, const uint8_t* __restrict__ wimg,
                float* __restrict__ out, double* __restrict__ stats) {
    using Cfg = DrCfg<CIN, COUT>;
    constexpr int G = DR_G;
    constexpr int GC = Cfg::GC;

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
            mbar_init(&full[s], DR_PRODUCERS / 32);      // one arrival per producer WARP
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
    if (warp >= 5 && warp < 9) {
        // accumulation is always "+=": start from zero accumulators
        const uint32_t taddr = tmem_base + ((uint32_t)((warp & 3) * 32) << 16);
        for (uint32_t c = 0; c < Cfg::TMEM_COLS; c += 8) tc_st8_zero(taddr + c);
        tc_wait_st();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();

    if (warp < 4) {
        // ===================== producers: global -> ring planes (cp.async, 16 B per op) =====================
        const int ptid = threadIdx.x;
        if (ptid == 0) {
            mbar_expect_tx(wbar, (uint32_t)p.wbytes);
            bulk_copy_g2s(wsm, wimg, (uint32_t)p.wbytes, wbar);
        }
        constexpr int NITEM = (Cfg::NKC * DR_NVOX + DR_PRODUCERS - 1) / DR_PRODUCERS;
        const int PF = p.pf;
        uint32_t slot = 0, sphase = 0, pslot = 0, pending = 0;
        const uint32_t ring_u32 = smem_u32(ring);
        auto publish = [&](int keep) {
            if (keep >= 7) asm volatile("cp.async.wait_group 7;" ::: "memory");
            else if (keep == 6) asm volatile("cp.async.wait_group 6;" ::: "memory");
            else if (keep == 5) asm volatile("cp.async.wait_group 5;" ::: "memory");
            else if (keep == 4) asm volatile("cp.async.wait_group 4;" ::: "memory");
            else if (keep == 3) asm volatile("cp.async.wait_group 3;" ::: "memory");
            else if (keep == 2) asm volatile("cp.async.wait_group 2;" ::: "memory");
            else if (keep == 1) asm volatile("cp.async.wait_group 1;" ::: "memory");
            else asm volatile("cp.async.wait_group 0;" ::: "memory");
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            __syncwarp();
            for (; pending > (uint32_t)keep; --pending) {
                if ((threadIdx.x & 31) == 0) mbar_arrive(&full[pslot]);
                if (++pslot == (uint32_t)R) pslot = 0;
            }
        };
        const size_t zstride_in = (size_t)p.H * p.W * CIN;
        DrIter units(p);
        DrUnit un;
        while (units.next(p, un)) {
            const int ibeg = un.z0 > 0 ? -1 : 0;
            int goff[NITEM];       // element offset inside a z plane, -1 = zero fill, -2 = no item
#pragma unroll
            for (int k = 0; k < NITEM; ++k) {
                const int j = ptid + k * DR_PRODUCERS;
                const int c = j % Cfg::NKC, v = j / Cfg::NKC;
                const int vy = v / DR_WW, vx = v - vy * DR_WW;
                const int gy = un.y0 - 1 + vy, gx = un.x0 - 1 + vx;
                const bool ok = gy >= 0 && gy < p.H && gx >= 0 && gx < p.W;
                goff[k] = (j >= Cfg::NKC * DR_NVOX) ? -2 : (ok ? (gy * p.W + gx) * CIN + c * 8 : -1);
            }
            const uint16_t* zbase = x + ((size_t)un.b * p.D + (un.z0 + ibeg)) * zstride_in;
            for (int i = ibeg; i < un.zlen; ++i, zbase += zstride_in) {
                mbar_wait(&empty[slot], sphase ^ 1);
                const uint32_t dst0 = ring_u32 + slot * (uint32_t)Cfg::SLOT_BYTES;
#pragma unroll
                for (int k = 0; k < NITEM; ++k) {
                    if (goff[k] != -2) {
                        const int j = ptid + k * DR_PRODUCERS;
                        const uint32_t soff = (uint32_t)((j % Cfg::NKC) * DR_KCH_PAD + (j / Cfg::NKC) * 16);
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
        // ===================== MMA issuer (one elected thread) =====================
        if (elect_one()) {
            mbar_wait(wbar, 0);
            tc_fence_after();
            constexpr uint32_t A_HI = (uint32_t)((DR_WW * 16) >> 4) | (1u << 14);          // SBO = next y row
            constexpr uint32_t B_HI = (uint32_t)(128 >> 4) | (1u << 14);                    // SBO = next 8 rows
            constexpr uint32_t A_LBO = (uint32_t)(DR_KCH_PAD >> 4) << 16;                   // next 8-channel chunk
            const uint32_t a_lo_ring = (smem_u32(ring) >> 4) | A_LBO;
            const uint32_t b_lo0 = (smem_u32(wsm) >> 4) | ((uint32_t)((Cfg::NROWS * 16) >> 4) << 16);
            auto issue_plane = [&](uint32_t dcol, uint32_t a_lo0, uint32_t b_lo, uint32_t idesc) {
#pragma unroll
                for (int s = 0; s < Cfg::NSTEPS; ++s) {
                    const int sh = s / Cfg::KS, ks = s % Cfg::KS;
                    // shift sh = (sy, sx) in {0,-1}^2: the tile origin sits at (1,1) of the halo plane
                    const int vy = 1 - (sh >> 1), vx = 1 - (sh & 1);
                    const uint32_t aoff = (uint32_t)((2 * ks * DR_KCH_PAD + (vy * DR_WW + vx) * 16) >> 4);
                    tc_mma_lohi1(dcol, a_lo0 + aoff, A_HI, b_lo + ((uint32_t)(s * Cfg::STEP_BYTES) >> 4), B_HI, idesc);
                }
            };
            uint32_t slot = 0, sphase = 0;
            uint32_t gq = 0, gphase = 0;       // accumulator group / phase of output plane t = 0 of the unit
            DrIter units(p);
            DrUnit un;
            while (units.next(p, un)) {
                const int ibeg = un.z0 > 0 ? -1 : 0;
                const int nt = 2 * un.zlen;
                uint32_t gw = gq, gwphase = gphase;   // group / phase of the next output plane to acquire
                int twaited = -1;
                uint32_t gdone = gq;
                for (int i = ibeg; i < un.zlen; ++i) {
                    // output planes (local t) this input plane feeds and the first row of its weight window
                    const int tlo = i < 0 ? 0 : 2 * i;
                    const int thi = i < 0 ? 0 : min(2 * i + 2, nt - 1);
                    const uint32_t wrow = i < 0 ? 2u * GC : 0u;
                    while (twaited < thi) {
                        mbar_wait(&tempty[gw], gwphase ^ 1);
                        ++twaited;
                        if (++gw == (uint32_t)G) { gw = 0; gwphase ^= 1; }
                    }
                    mbar_wait(&full[slot], sphase);
                    tc_fence_after();
                    const uint32_t a_lo0 = a_lo_ring + slot * (uint32_t)(Cfg::SLOT_BYTES >> 4);
                    uint32_t glo = gq + (uint32_t)tlo;
                    glo %= (uint32_t)G;
                    const int len = thi - tlo + 1;
                    const int len1 = min(len, G - (int)glo), len2 = len - len1;
                    issue_plane(tmem_base + glo * (uint32_t)GC, a_lo0, b_lo0 + ((wrow * 16u) >> 4),
                                ring_idesc(len1 * GC) | p.fmt);
                    if (len2 > 0)
                        issue_plane(tmem_base, a_lo0, b_lo0 + (((wrow + (uint32_t)(len1 * GC)) * 16u) >> 4),
                                    ring_idesc(len2 * GC) | p.fmt);
                    tc_commit(&empty[slot]);
                    if (++slot == (uint32_t)R) { slot = 0; sphase ^= 1; }
                    if (i >= 0) {
                        // output planes 2i and 2i+1 have received their last contribution
                        tc_commit(&tfull[gdone]);
                        if (++gdone == (uint32_t)G) gdone = 0;
                        tc_commit(&tfull[gdone]);
                        if (++gdone == (uint32_t)G) gdone = 0;
                    }
                }
                gq = gw; gphase = gwphase;
            }
        }
        __syncwarp();
    } else {
        // ===================== epilogue: 2 sets x 4 warps (128 TMEM lanes each) =====================
        const int set = (warp - 5) >> 2;          // warps 5-8: even output planes, warps 9-12: odd output planes
        const int g = warp & 3;                   // TMEM lane quarter of this warp
        const int row = g * 32 + lane;
        const int ty = row >> 3, tx = row & 7;
        float run[2 * COUT];
#pragma unroll
        for (int k = 0; k < 2 * COUT; ++k) run[k] = 0.f;
        float vmax = 0.f;
        const int vec = raw_vec_mode(out, COUT, COUT, 0);
        const bool fast16 = p.raw16 && (COUT % 8) == 0 && (((uintptr_t)out) & 31) == 0;
        const int Ho = 2 * p.H, Wo = 2 * p.W, Do = 2 * p.D;
        // a unit starts on an even group and consumes an even number of groups: set s only ever sees groups of parity s
        uint32_t grp = (uint32_t)set, gphase = 0;
        DrIter units(p);
        DrUnit un;
        while (units.next(p, un)) {
            const int y = un.y0 + ty, xq = un.x0 + tx;
            const bool ok = y < p.H && xq < p.W;
            const int nt = 2 * un.zlen;
            for (int t = set; t < nt; t += 2) {
                mbar_wait(&tfull[grp], gphase);
                tc_fence_after();
                const uint32_t taddr = tmem_base + ((uint32_t)(g * 32) << 16) + grp * (uint32_t)GC;
                uint64_t* const tempty_bar = &tempty[grp];
                grp += 2;
                if (grp >= (uint32_t)G) { grp -= (uint32_t)G; gphase ^= 1; }
                float v[GC];
#pragma unroll
                for (int c = 0; c < GC; c += 8) tc_ld8(taddr + c, v + c);
                tc_wait_ld();
#pragma unroll
                for (int c = 0; c < GC; c += 8) tc_st8_zero(taddr + c);
                tc_wait_st();
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(tempty_bar);
                if (!ok) continue;
                const int oz = 2 * un.z0 + t;
#pragma unroll
                for (int py = 0; py < 2; ++py) {
                    // classes (py, 0) and (py, 1) are x neighbours: 2 * Cout contiguous output values
                    const size_t off = ((((size_t)un.b * Do + oz) * Ho + (2 * y + py)) * Wo + 2 * xq) * COUT;
                    const float* vv = v + py * 2 * COUT;
                    if (fast16) {
#pragma unroll
                        for (int c = 0; c < 2 * COUT; c += 16) store_f16x16(reinterpret_cast<__half*>(out) + off + c, vv + c);
                    }
                    else store_raw_row<2 * COUT>(out, off, vv, 2 * COUT, vec, p.raw16, nullptr);
#pragma unroll
                    for (int c = 0; c < 2 * COUT; ++c) {
                        const float r = vv[c];
                        vmax = fmaxf(vmax, fabsf(r));
                        run[c % COUT] += r;
                        run[COUT + c % COUT] = fmaf(r, r, run[COUT + c % COUT]);
                    }
                }
            }
        }
        // fp16 raw output: count the threads that had to clamp a value (atvs_saturation_count)
        if (p.raw16 && p.sat != nullptr && vmax > 65504.f) atomicAdd(p.sat, 1ULL);
        if (stats != nullptr) {
#pragma unroll
            for (int k = 0; k < 2 * COUT; ++k) {
                float tot = run[k];
#pragma unroll
                for (int off = 16; off >= 1; off >>= 1) tot += __shfl_xor_sync(0xffffffffu, tot, off);
                if (lane == 0) atomicAdd(&stats[k], (double)tot);      // [sums (Cout) | sums of squares (Cout)]
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

// weight image: [shift (sy,sx) in {0,-1}^2][K=16 step][2 chunks][rows: kz0 | kz1 | kz2, each [class (py,px)][co]][8 ch]
// from the TF kernel [3,3,3,Cout,Cin]; (class, shift) pairs without a tap are zero rows
__global__ void k_pack_deconv_ring(const float* __restrict__ w, int Cin, int Cout, int f16, unsigned short* __restrict__ out) {
    const int ks_n = Cin / 16, gc = 4 * Cout, nrows = 3 * gc;
    const int sh = blockIdx.x / ks_n, ks = blockIdx.x % ks_n;
    const int sy = -(sh >> 1), sx = -(sh & 1);
    unsigned short* o = out + (size_t)blockIdx.x * 2 * nrows * 8;
    for (int i = threadIdx.x; i < 2 * nrows * 8; i += blockDim.x) {
        const int chunk = i / (nrows * 8), r = (i / 8) % nrows, e = i % 8;
        const int kz = r / gc, cls = (r % gc) / Cout, co = r % Cout;
        const int py = cls >> 1, px = cls & 1;
        // parity 0: taps (k=0, shift 0), (k=2, shift -1); parity 1: tap (k=1, shift 0)
        const int ky = py == 0 ? (sy == 0 ? 0 : 2) : (sy == 0 ? 1 : -1);
        const int kx = px == 0 ? (sx == 0 ? 0 : 2) : (sx == 0 ? 1 : -1);
        const int ci = (ks * 2 + chunk) * 8 + e;
        float val = 0.f;
        if (ky >= 0 && kx >= 0) val = w[((size_t)((kz * 3 + ky) * 3 + kx) * Cout + co) * Cin + ci];
        o[i] = tc_cvt16(val, f16);
    }
}

template <int CIN, int COUT>
int launch_dr(const uint16_t* x, const DrParams& p, const uint8_t* wimg, float* out, double* stats, size_t smem, int grid,
              cudaStream_t st) {
    if (const int rc = atvs_max_dynamic_smem<k_deconv3d_ring<CIN, COUT>>()) return rc;
    k_deconv3d_ring<CIN, COUT><<<grid, DR_THREADS, smem, st>>>(x, p, wimg, out, stats);
    ATVS_LAUNCH_CHECK();
    return 0;
}

size_t dr_wbytes(int Cin, int Cout) { return (size_t)4 * (Cin / 16) * 2 * (3 * 4 * Cout) * 16; }

}  // namespace

bool deconv_ring_supported(int Cin, int Cout) { return (Cin == 16 && Cout == 8) || (Cin == 32 && Cout == 16); }

bool deconv_ring_applicable(int B, int D, int H, int W) {
    // alone, the per-(class, tap) kernel is faster below ~100k input voxels (18.6 vs 30 us for 32 -> 16 on 32x32x40), but
    // inside the step the plane ring wins there too (5.93 vs 6.08 ms per cfg2 depth map: 110 KB of shared memory and 8
    // staged TMA tiles per 128 voxels less pressure on the co-running passes)
    return (long long)B * D * H * W >= 16384 && H >= 2 && W >= 2;
}

size_t deconv_ring_weight_bytes(int Cin, int Cout) {
    return deconv_ring_supported(Cin, Cout) ? (dr_wbytes(Cin, Cout) + 255) & ~(size_t)255 : 0;
}

int deconv_ring_pack(const float* kernel, int Cin, int Cout, int dtype, void* wimg, cudaStream_t st) {
    k_pack_deconv_ring<<<4 * (Cin / 16), 128, 0, st>>>(kernel, Cin, Cout, dtype == ATVS_F16, (unsigned short*)wimg);
    ATVS_LAUNCH_CHECK();
    return 0;
}

int deconv_ring(const void* x16, int dtype, const void* wimg, int B, int D, int H, int W, int Cin, int Cout, float* raw_out,
                int raw16, double* stats, cudaStream_t st) {
    const int sms = atvs_num_sms();
    DrParams p;
    memset(&p, 0, sizeof(p));
    p.B = B; p.D = D; p.H = H; p.W = W; p.Cout = Cout;
    p.raw16 = raw16;
    p.fmt = tc_fmt_bits(dtype);
    p.sat = raw16 ? atvs_sat_ptr() : nullptr;
    p.nXT = (W + DR_TX - 1) / DR_TX;
    p.nYT = (H + DR_TY - 1) / DR_TY;
    p.wbytes = (int)dr_wbytes(Cin, Cout);
    const size_t slot = ((size_t)(Cin / 8) * DR_KCH_PAD + 127) / 128 * 128;
    const size_t fixed = 128 + (size_t)((p.wbytes + 127) & ~127) + (2 * DR_MAXR + 2 * DR_G + 1) * 8 + 16;
    // one CTA of 13 warps per SM (8 epilogue warps need the registers); at most half of the shared memory, so that a
    // CTA of another stream's kernel can co-reside
    const int minb = 1;
    const size_t budget = 110 * 1024;
    int nring = (int)((budget - fixed) / slot);
    if (nring > 12) nring = 12;
    if (nring < 2) {
        atvs_set_error("atvs_conv3d_tc(deconv ring): weights do not fit next to 2 ring planes (Cin=%d Cout=%d)", Cin, Cout);
        return ATVS_E_UNSUP;
    }
    p.nring = nring;
    // planes of cp.async in flight per producer thread (the loads queue behind the kernel's own 8x larger write stream:
    // ~4000 cycles of latency in the timelines), at most nring - 1 and 8
    p.pf = nring - 1 < 8 ? nring - 1 : 8;
    p.total = (long long)B * p.nXT * p.nYT * D;
    const size_t smem = fixed + (size_t)nring * slot;
    const int grid = ring_balanced_grid(p.total, (long long)sms * minb, 20, 160);
    const uint8_t* wi = (const uint8_t*)wimg;
    if (Cin == 16 && Cout == 8) return launch_dr<16, 8>((const uint16_t*)x16, p, wi, raw_out, stats, smem, grid, st);
    if (Cin == 32 && Cout == 16) return launch_dr<32, 16>((const uint16_t*)x16, p, wi, raw_out, stats, smem, grid, st);
    atvs_set_error("atvs_conv3d_tc(deconv ring): no kernel for Cin=%d Cout=%d", Cin, Cout);
    return ATVS_E_UNSUP;
}
