// conv_ring.cu - stride-1 3x3x3 convolution (network.py:173-215 conv_bn, :142 conv) as a
// tcgen05 implicit GEMM over a shared-memory RING OF HALO PLANES, z-EXPANDED in the MMA N dimension.
//
// What bounds a Cout = 8 convolution on the tensor pipe is the fetch of the A operand (the voxel
// tile) from shared memory: tools/mma_probe.cu measures  t(M=128, N, K=16) = 32 + N/4 cycles  with both
// operands in shared memory (A = 4 KB at 128 B/clk, B = 32 N bytes), i.e. N = 16 costs 39 cycles
// while its math needs 8.  So every fetched A tile has to feed as many output columns as possible.
// The three z taps of a 3x3x3 kernel see the SAME in-plane tile: input plane i (shifted by the
// in-plane tap (dy,dx)) contributes to the output planes i-2, i-1, i with the weights dz = 2, 1, 0.
// One MMA therefore covers three output planes:
//
//   accumulators  : a ring of G column groups in TMEM, one group (CP = 8|16|32 columns) per output plane
//   per input plane: 9 * Cin/16 MMAs (5 tap-pair MMAs for Cin = 8) with N = 3*CP over three consecutive
//                    groups and B = [w_dz2 | w_dz1 | w_dz0]; the plane is consumed ONCE and its ring
//                    slot released, an output plane is complete after the input plane behind it
//   -> 3x fewer MMAs than one accumulator per output plane (N = CP), each ~ the same cost.
//
// N must be a multiple of 16: with CP = 8 an odd run of groups is extended by one group that meets
// zero weights (the next, already drained and zeroed group, or a never-read dummy group behind the
// ring); runs that wrap around the ring are issued as two MMAs.  Accumulation is always "+=": the
// epilogue zeroes a group (tcgen05.st) right after reading it.
//
//   work unit : a column of 16(y) x 8(x) output tiles over a z segment [z0, z0+zlen)
//   ring slot : one input z plane with halo, [Cin/8 chunks][18 y][10 x][8 channels] bf16, no-swizzle
//               K-major core matrices (8 consecutive x = one 8-row core matrix, next y row = SBO, next
//               8-channel chunk = LBO), filled by 4 producer warps with 16-byte cp.async (zero fill =
//               'SAME' padding) and published to the async proxy with fence.proxy.async
//   Cin = 8   : one K=16 step covers two taps of the plane (LBO = distance of the taps)
//   warps 0-3 producers | warp 4 MMA issuer (one elected lane) | warps 5-8 epilogue
//
// The issuing thread's stream is ~10 SASS instructions per MMA (descriptor arithmetic in vector registers + R2UR moves
// to the uniform registers UTCHMMA reads) and sustains one MMA per ~47 cycles against the pipe's 40
// (profiles/r02_ring32_issue_trace.txt).  Splitting the two MMA tiles of a plane over two issuing warps (4 and 9, each
// committing its own MMAs) was built and measured: 93.7 us against 93.9 for 32 -> 8, 51.2 against 48.7 for 8 -> 8 at
// cfg2 - the pipe, not the issue stream, is what the plane step waits for; one issuer stays.
#include "ring_common.cuh"
#include "conv_ring.cuh"
#include <cstring>

namespace {


// one CTA plane = RG_MT = 2 MMA tiles (16 y x 8 x each) side by side in x: 256 voxels per plane step, published as one
// cp.async group.  The skeleton of the three roles (no loads / MMAs / stores) runs at ~760 cycles per 256-voxel plane
// (profiles/r02_ring_8_8_trace.txt), which is what bounds the 8-channel layers; 4-tile planes (512 voxels, 7-group
// accumulator ring so that two CTAs still share the 512 TMEM columns) and grouped publishing of 2-4 planes were built to
// amortise it and measured: neither changes the 45 us of an 8 -> 8 layer at cfg2 (profiles/r02_ring_probe.txt), so the
// cost scales with the plane, not with the handshake count.
constexpr int RG_TY = 16, RG_HH = RG_TY + 2;
constexpr int RG_MT = 2, RG_TX = 8 * RG_MT, RG_WW = RG_TX + 2;
constexpr int RG_PRODUCERS = 128;
constexpr int RG_THREADS = 288;
constexpr int RG_MAXG = 15;
constexpr int RG_MAXR = 16;      // mbarrier pairs reserved for the ring slots

struct RingParams {
    int B, D, H, W;
    int Cout, coff, ncols;
    int raw16;          // raw output dtype: 0 fp32, 1 saturated fp16
    uint32_t fmt;       // operand format bits of the instruction descriptor (tc_fmt_bits)
    unsigned long long* sat;   // saturation counter of the fp16 raw stores (atvs_sat_ptr)
    int nXT, nYT;
    int nring, pf;      // ring slots; planes of cp.async in flight per producer thread (pf < nring)
    int wbytes;
    long long total;    // tile columns * D: the plane sequence cut into one range per CTA (RingSpan)
};

template <int CIN, int CP>
struct RingCfg {
    static constexpr int NVOX = RG_HH * RG_WW;            // voxels of one halo plane (324)
    static constexpr int KCH_PAD = NVOX * 16 + 16;        // pitch of one 8-channel chunk plane; +16 B keeps the
                                                          // 8 chunk stores of a voxel on distinct banks
    static constexpr int NKC = CIN / 8;
    static constexpr int SLOT_BYTES = (NKC * KCH_PAD + 127) / 128 * 128;
    static constexpr int NSTEPS = (CIN >= 16) ? 9 * (CIN / 16) : 5;     // K=16 MMA steps per input plane
    static constexpr bool PAD = (CP == 8);                              // runs are padded to N % 16 == 0 with zero weights
    static constexpr int G = (CP == 8) ? 15 : 8;                        // accumulator groups in the ring
    static constexpr int NROWS = (CP == 8) ? 64 : 3 * CP;               // rows of one weight step image
    static constexpr int STEP_BYTES = 2 * NROWS * 16;
    static constexpr uint32_t TILE_COLS = (CP == 32) ? 256u : 128u;    // CP=8: G groups + 1 dummy
    static constexpr uint32_t TMEM_COLS = RG_MT * TILE_COLS;
};

struct Unit {
    int b, x0, y0, z0, zlen;
};


// units of this CTA (ring_common.cuh RingSpan: one balanced range of the plane sequence)
struct UnitIter {
    RingSpan span;
    __device__ __forceinline__ explicit UnitIter(const RingParams& p) : span(p.total) {}
    __device__ __forceinline__ bool next(const RingParams& p, Unit& r) {
        long long t;
        if (!span.next(p.D, t, r.z0, r.zlen)) return false;
        r.x0 = (int)(t % p.nXT) * RG_TX;
        t /= p.nXT;
        r.y0 = (int)(t % p.nYT) * RG_TY;
        r.b = (int)(t / p.nYT);
        return true;
    }
};

// input planes of a unit: i in [ibeg, iend], plane i = volume plane z0 - 1 + i; planes outside the volume
// contribute nothing ('SAME' zero padding) and are skipped by all three roles
__device__ __forceinline__ int unit_ibeg(const Unit& u) { return u.z0 == 0 ? 1 : 0; }
__device__ __forceinline__ int unit_iend(const RingParams& p, const Unit& u) {
    return (u.z0 + u.zlen == p.D) ? u.zlen : u.zlen + 1;
}

// weight-image window (in rows of 8) and MMA N for a run of `len` output planes whose first plane meets
// the z tap `f` (2, 1 or 0; the following planes meet f-1, ...).
//   CP = 8 image groups : [w2 0 w1 0 w2 w1 w0 0]      CP = 16, 32 : [w2 w1 w0]
template <int CP>
__device__ __forceinline__ void ring_window(int f, int len, uint32_t& row_off_bytes, uint32_t& idesc) {
    if (CP == 8) {
        int grp;
        if (len == 1) grp = (f == 2) ? 0 : (f == 1 ? 2 : 6);
        else if (len == 2) grp = (f == 2) ? 4 : 5;
        else grp = 4;
        row_off_bytes = (uint32_t)grp * 128u;
        idesc = ring_idesc(len == 3 ? 32 : 16);
    } else {
        row_off_bytes = (uint32_t)(2 - f) * (uint32_t)CP * 16u;
        idesc = ring_idesc(len * CP);
    }
}

template <int CIN, int CP, int MINB, bool FAST>
__global__ void __launch_bounds__(RG_THREADS, MINB)
k_conv3d_ring(const uint16_t* __restrict__ x, const __grid_constant__ RingParams p,
              const uint8_t* __restrict__ wimg, float* __restrict__ out, double* __restrict__ stats,
              const float* __restrict__ bias) {
    using Cfg = RingCfg<CIN, CP>;
    constexpr int G = Cfg::G;
    constexpr int RG_NVOX = Cfg::NVOX, RG_KCH_PAD = Cfg::KCH_PAD;

    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>(((uintptr_t)smem_raw + 127) & ~(uintptr_t)127);
    uint8_t* wsm = smem;
    uint8_t* ring = smem + ((p.wbytes + 127) & ~127);
    uint64_t* bars = reinterpret_cast<uint64_t*>(ring + (size_t)p.nring * Cfg::SLOT_BYTES);
    uint64_t* full = bars;
    uint64_t* empty = bars + p.nring;
    uint64_t* tfull = bars + 2 * p.nring;
    uint64_t* tempty = tfull + RG_MAXG;
    uint64_t* wbar = tempty + RG_MAXG;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(wbar + 1);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int R = p.nring;
    if (threadIdx.x == 0) {
        for (int s = 0; s < R; ++s) {
            mbar_init(&full[s], RG_PRODUCERS / 32);      // one arrival per producer WARP (lane 0, after __syncwarp)
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
        // ===================== producers: global -> ring planes (cp.async, 16 B per op) =====================
        const int ptid = threadIdx.x;
        if (ptid == 0) {
            mbar_expect_tx(wbar, (uint32_t)p.wbytes);
            bulk_copy_g2s(wsm, wimg, (uint32_t)p.wbytes, wbar);
        }
        // this thread's share of a halo plane: items j = ptid + k*128 -> (chunk c, halo voxel v).  The
        // shared-memory offsets never change and the global offsets change once per unit, so one plane
        // costs a handful of instructions per item.
        constexpr int NITEM = (Cfg::NKC * RG_NVOX + RG_PRODUCERS - 1) / RG_PRODUCERS;
        // up to PF planes of cp.async in flight per thread; plane q is published (fence.proxy.async +
        // mbarrier arrive) once plane q+PF-1 has been issued.  PF <= R-1 keeps the ring deadlock-free.
        // Publishing a plane (cp.async.wait_group + fence.proxy.async + __syncwarp + mbarrier arrive) costs ~400 cycles of
        // the producer's per-plane loop whatever the plane holds (profiles/r02_ring_8_8_trace.txt: 770 cycles per plane
        // with nothing to load).
        const int PF = p.pf;      // 1..4
        uint32_t slot = 0, sphase = 0, pslot = 0, pending = 0;
        const uint32_t ring_u32 = smem_u32(ring);
        auto publish = [&](int keep) {
            // wait until at most `keep` planes are pending, then publish every older plane
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
        UnitIter units(p);
        Unit un;
        while (units.next(p, un)) {
            const int ibeg = unit_ibeg(un), iend = unit_iend(p, un);
            int goff[NITEM];       // element offset inside a z plane, -1 = zero fill, -2 = no item
#pragma unroll
            for (int k = 0; k < NITEM; ++k) {
                const int j = ptid + k * RG_PRODUCERS;
                const int c = j % Cfg::NKC, v = j / Cfg::NKC;
                const int vy = v / RG_WW, vx = v - vy * RG_WW;
                const int gy = un.y0 - 1 + vy, gx = un.x0 - 1 + vx;
                const bool ok = gy >= 0 && gy < p.H && gx >= 0 && gx < p.W;
                goff[k] = (j >= Cfg::NKC * RG_NVOX) ? -2 : (ok ? (gy * p.W + gx) * CIN + c * 8 : -1);
            }
            const uint16_t* zbase = x + ((size_t)un.b * p.D + (un.z0 - 1 + ibeg)) * zstride_in;
            for (int i = ibeg; i <= iend; ++i, zbase += zstride_in) {
                mbar_wait(&empty[slot], sphase ^ 1);
                const uint32_t dst0 = ring_u32 + slot * (uint32_t)Cfg::SLOT_BYTES;
#pragma unroll
                for (int k = 0; k < NITEM; ++k) {
                    if (goff[k] != -2) {
                        const int j = ptid + k * RG_PRODUCERS;
                        const uint32_t soff = (uint32_t)((j % Cfg::NKC) * RG_KCH_PAD + (j / Cfg::NKC) * 16);
                        const bool ok = goff[k] >= 0;
                        const uint16_t* src = ok ? zbase + goff[k] : x;
                        asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst0 + soff), "l"(src),
                                     "r"(ok ? 16 : 0)
                                     : "memory");
                    }
                }
                if (++slot == (uint32_t)R) { slot = 0; sphase ^= 1; }
                asm volatile("cp.async.commit_group;" ::: "memory");
                if (++pending >= (uint32_t)PF) publish(PF - 1);
            }
        }
        publish(0);
    } else if (warp == 4) {
        // ===================== MMA issuer (elected lane) =====================
        // The instruction stream per plane matters for the small-channel layers: counters are incremental (no
        // divisions), and the steady state (three live output planes, no ring wrap) is a straight-line block.
        if (elect_one()) {
        mbar_wait(wbar, 0);
        tc_fence_after();
        constexpr uint32_t A_HI = (uint32_t)((RG_WW * 16) >> 4) | (1u << 14);          // SBO = next y row
        constexpr uint32_t B_HI = (uint32_t)(128 >> 4) | (1u << 14);                    // SBO = next 8 rows
        constexpr uint32_t A_LBO = (CIN >= 16) ? ((uint32_t)(RG_KCH_PAD >> 4) << 16) : 0u;
        constexpr uint32_t FAST_BOFF = (CP == 8) ? 4u * 128u : 0u;                      // window [w2 w1 w0 (0)]
        const uint32_t FAST_IDESC = ring_idesc(CP == 8 ? 32 : 3 * CP) | p.fmt;
        const uint32_t a_lo_ring = (smem_u32(ring) >> 4) | A_LBO;
        const uint32_t b_lo0 = (smem_u32(wsm) >> 4) | ((uint32_t)((Cfg::NROWS * 16) >> 4) << 16);
        auto issue_plane = [&](uint32_t dcol, uint32_t a_lo0, uint32_t b_lo, uint32_t idesc) {
#pragma unroll
            for (int s = 0; s < Cfg::NSTEPS; ++s) {
                uint32_t aoff;
                if (CIN >= 16) {
                    constexpr int KS = (CIN >= 16) ? CIN / 16 : 1;
                    const int tp = s / KS, ks = s % KS;
                    aoff = (uint32_t)((2 * ks * RG_KCH_PAD + ((tp / 3) * RG_WW + (tp % 3)) * 16) >> 4);
                } else {
                    // tap pairs (0,1) (2,3) (4,5) (6,7) (7*,8): the 9th tap is paired with a second,
                    // zero-weighted read of tap 7 so that every operand byte is real data
                    const int ta = (s < 4) ? 2 * s : 7, tb = (s < 4) ? 2 * s + 1 : 8;
                    const uint32_t offa = (uint32_t)(((ta / 3) * RG_WW + (ta % 3)) * 16);
                    const uint32_t offb = (uint32_t)(((tb / 3) * RG_WW + (tb % 3)) * 16);
                    aoff = (offa >> 4) | (((offb - offa) >> 4) << 16);
                }
#pragma unroll
                for (int mt = 0; mt < RG_MT; ++mt)
                    tc_mma_lohi1(dcol + (uint32_t)mt * Cfg::TILE_COLS, a_lo0 + aoff + (uint32_t)(mt * 8), A_HI,
                                 b_lo + ((uint32_t)(s * Cfg::STEP_BYTES) >> 4), B_HI, idesc);
            }
        };
        uint32_t slot = 0, sphase = 0;     // ring position of the next input plane
        uint32_t gq = 0, gphase = 0;       // accumulator group / phase of output plane t = 0 of the unit
        UnitIter units(p);
        Unit un;
        while (units.next(p, un)) {
            const int ibeg = unit_ibeg(un), iend = unit_iend(p, un);
            uint32_t gw = gq, gwphase = gphase;   // group / phase of the next output plane to wait for
            int twaited = -1;
            uint32_t glo = gq;                    // group of output plane max(0, i - 2)
            uint32_t gdone = gq;                  // group of the next output plane to complete
            int tdone = 0;
            for (int i = ibeg; i <= iend; ++i) {
                const int tlo = max(0, i - 2), thi = min(un.zlen - 1, i);
                // accumulator groups of the run; the group behind it may be touched with zero weights
                // (CP = 8), so it must have been drained as well
                const int tneed = thi + (Cfg::PAD ? 1 : 0);
                while (twaited < tneed) {
                    mbar_wait(&tempty[gw], gwphase ^ 1);
                    ++twaited;
                    if (++gw == (uint32_t)G) { gw = 0; gwphase ^= 1; }
                }
                mbar_wait(&full[slot], sphase);
                tc_fence_after();
                const uint32_t a_lo0 = a_lo_ring + slot * (uint32_t)(Cfg::SLOT_BYTES >> 4);
                if (thi - tlo == 2 && glo + 3 <= (uint32_t)G) {
                    issue_plane(tmem_base + glo * (uint32_t)CP, a_lo0, b_lo0 + (FAST_BOFF >> 4), FAST_IDESC);
                } else {
                    const int len = thi - tlo + 1, f = i - tlo;
                    const int len1 = min(len, G - (int)glo), len2 = len - len1;
                    uint32_t boff, idesc;
                    ring_window<CP>(f, len1, boff, idesc);
                    issue_plane(tmem_base + glo * (uint32_t)CP, a_lo0, b_lo0 + (boff >> 4), idesc | p.fmt);
                    if (len2 > 0) {
                        ring_window<CP>(f - len1, len2, boff, idesc);
                        issue_plane(tmem_base, a_lo0, b_lo0 + (boff >> 4), idesc | p.fmt);
                    }
                }
                tc_commit(&empty[slot]);
                if (++slot == (uint32_t)R) { slot = 0; sphase ^= 1; }
                if (i >= 2 && ++glo == (uint32_t)G) glo = 0;
                // output planes whose last contribution this was: t <= i - 2, and all of them at the end
                const int tlast = (i == iend) ? un.zlen - 1 : i - 2;
                while (tdone <= tlast) {
                    tc_commit(&tfull[gdone]);
                    ++tdone;
                    if (++gdone == (uint32_t)G) gdone = 0;
                }
            }
            gq = gw; gphase = gwphase;
            if (twaited >= un.zlen) {      // the CP = 8 look-ahead waited for the next unit's first plane
                gq = (gq == 0) ? (uint32_t)G - 1 : gq - 1;
                if (gq == (uint32_t)G - 1) gphase ^= 1;
            }
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
        // the CRM's layers: full slab of CP columns, saturated fp16 rows of whole 16-byte groups.  Their plane step is bound by
        // this warp's instruction stream (one epilogue warp per SM sub-partition and CTA: ~270 dependent instructions per
        // plane through the generic row store with its per-column predicates and 64-bit index arithmetic), so they take a
        // straight-line path: no column predicates, row pointer carried from plane to plane.
        constexpr bool fast = FAST;      // host: ncols == CP, 32-byte aligned fp16 rows (ring_conv)
        uint32_t grp = 0, gphase = 0;
        UnitIter units(p);
        Unit un;
        while (units.next(p, un)) {
            const int y = un.y0 + ty, xq = un.x0 + tx;          // tile mt covers x = xq + 8 * mt
            const bool yok = y < p.H;
            const size_t obase = ((((size_t)un.b * p.D + un.z0) * p.H + (yok ? y : 0)) * p.W) * p.Cout + p.coff;
            const size_t zstride = (size_t)p.H * p.W * p.Cout;
            __half* orow16 = reinterpret_cast<__half*>(out) + obase + (size_t)xq * p.Cout;    // fast path: this thread's row, plane t
            // depth-invariant part of the layer (the tiled reference-feature half of the cost volume): the interior-plane
            // class is the same for all but the first and last plane of the volume - fetched once per unit
            // (8-channel layers only: wider accumulator rows would spill)
            constexpr bool HOIST = (CP == 8);
            float bint[HOIST ? RG_MT : 1][HOIST ? CP : 1];
            if (HOIST && bias != nullptr && yok) {
#pragma unroll
                for (int mt = 0; mt < RG_MT; ++mt) {
                    const int xm = xq + 8 * mt;
                    const float* brow = bias + ((((size_t)un.b * 3 + 1) * p.H + y) * p.W + (xm < p.W ? xm : 0)) * p.Cout + p.coff;
#pragma unroll
                    for (int c = 0; c < CP; ++c) bint[mt][c] = (c < p.ncols) ? __ldg(brow + c) : 0.f;
                }
            }
            for (int t = 0; t < un.zlen; ++t) {
                mbar_wait(&tfull[grp], gphase);
                tc_fence_after();
                const uint32_t taddr = tmem_base + ((uint32_t)(g * 32) << 16) + grp * (uint32_t)CP;
                uint64_t* const tempty_bar = &tempty[grp];
                if (++grp == (uint32_t)G) { grp = 0; gphase ^= 1; }
                float v[RG_MT][CP];
#pragma unroll
                for (int mt = 0; mt < RG_MT; ++mt)
#pragma unroll
                    for (int c = 0; c < CP; c += 8) tc_ld8(taddr + (uint32_t)mt * Cfg::TILE_COLS + c, v[mt] + c);
                tc_wait_ld();
#pragma unroll
                for (int mt = 0; mt < RG_MT; ++mt)
#pragma unroll
                    for (int c = 0; c < CP; c += 8) tc_st8_zero(taddr + (uint32_t)mt * Cfg::TILE_COLS + c);
                // release the group before the plane is converted and stored (releasing it after the stores, with the
                // zeroing overlapped with the conversion, measured 31.7 vs 31.9 us per 8 -> 8 layer in steady state)
                __syncwarp();
                tc_wait_st();
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(tempty_bar);
                if (FAST && yok) {
                    const int z = un.z0 + t;
                    const int zc = (z == 0) ? 0 : (z == p.D - 1 ? 2 : 1);
#pragma unroll
                    for (int mt = 0; mt < RG_MT; ++mt) {
                        const int xm = xq + 8 * mt;
                        if (xm < p.W) {
                            if (bias != nullptr) {
                                if (HOIST && zc == 1) {
#pragma unroll
                                    for (int c = 0; c < CP; ++c) v[mt][c] += bint[HOIST ? mt : 0][HOIST ? c : 0];
                                } else {
                                    const float4* brow = reinterpret_cast<const float4*>(
                                        bias + ((((size_t)un.b * 3 + zc) * p.H + y) * p.W + xm) * p.Cout + p.coff);
#pragma unroll
                                    for (int c = 0; c < CP; c += 4) {
                                        const float4 bv = __ldg(brow + (c >> 2));
                                        v[mt][c] += bv.x; v[mt][c + 1] += bv.y; v[mt][c + 2] += bv.z; v[mt][c + 3] += bv.w;
                                    }
                                }
                            }
                            float m = fabsf(v[mt][0]);
#pragma unroll
                            for (int c = 1; c < CP; ++c) m = fmaxf(m, fabsf(v[mt][c]));
                            if (m > 65504.f) atomicAdd(p.sat, 1ULL);
                            __half* op = orow16 + mt * 8 * p.Cout;
#pragma unroll
                            for (int c = 0; c < CP; c += 8) {
                                uint4 u;
                                u.x = pack_f16x2_sat(v[mt][c], v[mt][c + 1]); u.y = pack_f16x2_sat(v[mt][c + 2], v[mt][c + 3]);
                                u.z = pack_f16x2_sat(v[mt][c + 4], v[mt][c + 5]); u.w = pack_f16x2_sat(v[mt][c + 6], v[mt][c + 7]);
                                *reinterpret_cast<uint4*>(op + c) = u;
                            }
                            if (stats != nullptr) {
#pragma unroll
                                for (int c = 0; c < CP; ++c) {
                                    run[c] += v[mt][c];
                                    run[CP + c] = fmaf(v[mt][c], v[mt][c], run[CP + c]);
                                }
                            }
                        }
                    }
                } else if (!FAST && yok) {
                const int z = un.z0 + t;
                const int zc = (z == 0) ? 0 : (z == p.D - 1 ? 2 : 1);
#pragma unroll
                for (int mt = 0; mt < RG_MT; ++mt) {
                    const int xm = xq + 8 * mt;
                    if (xm >= p.W) continue;
                    const size_t ooff = obase + (size_t)t * zstride + (size_t)xm * p.Cout;
                    if (HOIST && bias != nullptr && zc == 1) {
#pragma unroll
                        for (int c = 0; c < CP; ++c) v[mt][c] += bint[HOIST ? mt : 0][HOIST ? c : 0];
                    } else if (bias != nullptr) {
                        const float* brow = bias + ((((size_t)un.b * 3 + zc) * p.H + y) * p.W + xm) * p.Cout + p.coff;
                        if (vec4) {
#pragma unroll
                            for (int c = 0; c < CP; c += 4)
                                if (c < p.ncols) {
                                    const float4 bv = __ldg(reinterpret_cast<const float4*>(brow + c));
                                    v[mt][c] += bv.x; v[mt][c + 1] += bv.y; v[mt][c + 2] += bv.z; v[mt][c + 3] += bv.w;
                                }
                        } else {
#pragma unroll
                            for (int c = 0; c < CP; ++c)
                                if (c < p.ncols) v[mt][c] += __ldg(brow + c);
                        }
                    }
                    store_raw_row<CP>(out, ooff, v[mt], p.ncols, vec, p.raw16, p.sat);
                    if (stats != nullptr) {
                        // per-THREAD running moments (rows = this thread's voxels): no cross-lane traffic per tile
#pragma unroll
                        for (int c = 0; c < CP; ++c) {
                            run[c] += v[mt][c];
                            run[CP + c] = fmaf(v[mt][c], v[mt][c], run[CP + c]);
                        }
                    }
                }
                }
                orow16 += zstride;
            }
        }
        if (stats != nullptr) {
            // [sums | sums of squares] of this thread -> warp totals -> fp64 atomics
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

// weight image of one Cout slab: [step][2 chunks][NROWS rows][8 channels] 16-bit; the rows are groups of
// CP output channels, each group holding one z tap (or zeros), see ring_window()
__global__ void k_pack_ring(const float* __restrict__ w, int Cin, int Cout, int cp, int nslabs, int f16,
                            unsigned short* __restrict__ out) {
    const int nsteps = ring_nsteps(Cin);
    const int nrows = (cp == 8) ? 64 : 3 * cp;
    const int slab = blockIdx.x / nsteps, step = blockIdx.x % nsteps;
    unsigned short* o = out + ((size_t)slab * nsteps + step) * 2 * nrows * 8;
    for (int i = threadIdx.x; i < 2 * nrows * 8; i += blockDim.x) {
        const int chunk = i / (nrows * 8), r = (i / 8) % nrows, e = i % 8;
        const int grp = r / cp, n = r % cp;
        int dz;
        if (cp == 8) {
            const int map[8] = {2, -1, 1, -1, 2, 1, 0, -1};
            dz = map[grp];
        } else {
            dz = 2 - grp;
        }
        int tap2d, k;
        if (Cin >= 16) {
            tap2d = step / (Cin / 16);
            k = ((step % (Cin / 16)) * 2 + chunk) * 8 + e;
        } else {
            // pairs (0,1) (2,3) (4,5) (6,7) (7*,8): chunk 0 of the last pair is a zero-weighted re-read of tap 7
            tap2d = (step < 4) ? 2 * step + chunk : (chunk == 0 ? -1 : 8);
            k = e;
        }
        const int co = slab * cp + n;
        float val = 0.f;
        if (dz >= 0 && tap2d >= 0 && co < Cout) val = w[((size_t)(dz * 9 + tap2d) * Cin + k) * Cout + co];
        o[i] = tc_cvt16(val, f16);
    }
}

template <int CIN, int CP, int MINB, bool FAST>
int launch_ring1(const uint16_t* x, const RingParams& p, const uint8_t* wimg, float* out, double* stats,
                 const float* bias, size_t smem, int grid, cudaStream_t st) {
    if (const int rc = atvs_max_dynamic_smem<k_conv3d_ring<CIN, CP, MINB, FAST>>()) return rc;
    k_conv3d_ring<CIN, CP, MINB, FAST><<<grid, RG_THREADS, smem, st>>>(x, p, wimg, out, stats, bias);
    ATVS_LAUNCH_CHECK();
    return 0;
}

// FAST epilogue: the slab fills its CP columns and the rows are saturated fp16 in whole, 32-byte aligned groups of 8
template <int CIN, int CP, int MINB>
int launch_ring(const uint16_t* x, const RingParams& p, const uint8_t* wimg, float* out, double* stats,
                const float* bias, size_t smem, int grid, cudaStream_t st) {
    const bool fast = p.ncols == CP && p.raw16 && ((p.Cout | p.coff) & 7) == 0 && (((uintptr_t)out) & 31) == 0 &&
                      (bias == nullptr || (((uintptr_t)bias) & 15) == 0);
    return fast ? launch_ring1<CIN, CP, MINB, true>(x, p, wimg, out, stats, bias, smem, grid, st)
                : launch_ring1<CIN, CP, MINB, false>(x, p, wimg, out, stats, bias, smem, grid, st);
}

size_t ring_slab_bytes(int Cin, int cp) {
    return (size_t)ring_nsteps(Cin) * 2 * ((cp == 8) ? 64 : 3 * cp) * 16;
}

}  // namespace

// columns per output plane: the smallest of {8, 16, 32} covering Cout (more output channels: slabs of 32)
int ring_npad(int Cin, int Cout) {
    (void)Cin;
    return Cout <= 8 ? 8 : Cout <= 16 ? 16 : 32;
}

size_t ring_weight_bytes(int Cin, int Cout) {
    const int cp = ring_npad(Cin, Cout);
    const int nslabs = (Cout + cp - 1) / cp;
    return (size_t)nslabs * ring_slab_bytes(Cin, cp);
}

int ring_pack(const float* kernel, int Cin, int Cout, int dtype, void* wimg, cudaStream_t st) {
    const int cp = ring_npad(Cin, Cout);
    const int nslabs = (Cout + cp - 1) / cp;
    k_pack_ring<<<nslabs * ring_nsteps(Cin), 128, 0, st>>>(kernel, Cin, Cout, cp, nslabs, dtype == ATVS_F16,
                                                           (unsigned short*)wimg);
    ATVS_LAUNCH_CHECK();
    return 0;
}

bool ring_applicable(int B, int D, int H, int W, int stride, int transposed) {
    // smaller volumes: the per-tap TMA kernel (conv_tc.cu).  Alone it is as fast there, but it fetches every input voxel 27
    // times through L2 and spends 5 x the SM time of the ring on a 32 -> 32 layer of 32x32x40 voxels: inside the step the
    // ring wins from ~32k voxels (5.21 -> 5.05 ms per cfg2 depth map with the threshold lowered from 65536)
    return !transposed && stride == 1 && (long long)D * H * W >= 32768 && H >= 8 && W >= 8;
}

int ring_conv(const void* x16, int dtype, const void* wimg, int B, int D, int H, int W, int Cin, int Cout, float* raw_out,
              int raw16, double* stats, const float* bias, cudaStream_t st) {
    const int cp = ring_npad(Cin, Cout);
    const int nslabs = (Cout + cp - 1) / cp;
    const int sms = atvs_num_sms();
    RingParams p;
    memset(&p, 0, sizeof(p));
    p.B = B; p.D = D; p.H = H; p.W = W; p.Cout = Cout;
    p.raw16 = raw16;
    p.fmt = tc_fmt_bits(dtype);
    p.sat = raw16 ? atvs_sat_ptr() : nullptr;
    p.nXT = (W + RG_TX - 1) / RG_TX;
    p.nYT = (H + RG_TY - 1) / RG_TY;
    p.wbytes = (int)ring_slab_bytes(Cin, cp);
    const size_t slot = ((size_t)(Cin / 8) * ((size_t)RG_HH * RG_WW * 16 + 16) + 127) / 128 * 128;
    const size_t fixed = 128 + (size_t)((p.wbytes + 127) & ~127) + (2 * RG_MAXR + 2 * RG_MAXG + 1) * 8 + 16;
    // two co-resident CTAs per SM when 2 x (weights + 4 planes) fit: their producer / MMA / epilogue
    // handshake latencies overlap
    int minb = (cp < 32 && fixed + 3 * slot <= 110 * 1024) ? 2 : 1;
    // small volumes: a second CTA per SM only halves the few plane steps each CTA gets, while every CTA pays
    // the same cold start (measured 41 -> 29 us for 16->16 on 64x64x80)
    if ((long long)B * p.nXT * p.nYT * D < (long long)sms * 2 * 12) minb = 1;
    const size_t budget = (minb == 2 ? 110 : 220) * 1024;
    int nring = (int)((budget - fixed) / slot);
    if (nring > 8) nring = 8;
    if (nring < 2) {
        atvs_set_error("atvs_conv3d_bf16(ring): weights do not fit next to 2 ring planes (Cin=%d Cout=%d)", Cin, Cout);
        return ATVS_E_UNSUP;
    }
    p.nring = nring;
    p.pf = nring - 1 < 4 ? nring - 1 : 4;          // planes in flight: pf < nring keeps the ring deadlock-free
    p.total = (long long)B * p.nXT * p.nYT * D;
    const size_t smem = fixed + (size_t)nring * slot;
    const int grid = ring_balanced_grid(p.total, (long long)sms * minb, 12, 40);
    for (int slab = 0; slab < nslabs; ++slab) {
        p.coff = slab * cp;
        p.ncols = (Cout - p.coff < cp) ? Cout - p.coff : cp;
        const uint8_t* wi = (const uint8_t*)wimg + (size_t)slab * p.wbytes;
        int rc = 0;
#define RG_CASE(CI, CPV)                                                                                              \
    if (Cin == CI && cp == CPV) {                                                                                     \
        rc = (minb == 2) ? launch_ring<CI, CPV, 2>((const uint16_t*)x16, p, wi, raw_out, stats, bias, smem, grid, st) \
                         : launch_ring<CI, CPV, 1>((const uint16_t*)x16, p, wi, raw_out, stats, bias, smem, grid, st); \
    } else
        RG_CASE(8, 8) RG_CASE(8, 16) RG_CASE(8, 32) RG_CASE(16, 8) RG_CASE(16, 16) RG_CASE(16, 32)
        RG_CASE(32, 8) RG_CASE(32, 16) RG_CASE(32, 32) RG_CASE(64, 8) RG_CASE(64, 16) RG_CASE(64, 32)
        {
            atvs_set_error("atvs_conv3d_bf16(ring): no kernel for Cin=%d CP=%d", Cin, cp);
            return ATVS_E_UNSUP;
        }
#undef RG_CASE
        if (rc) return rc;
    }
    return 0;
}
