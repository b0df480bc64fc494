// conv_attn_ring.cu - attention aggregation module (network.py:282-351 attention_activation + :379-408
// attention_aggregation) as ONE kernel: K2 without its logits in HBM.
//
// Per view n the reference evaluates two 3x3x3 8 -> 8 convolutions with weights shared by all views,
//   u_n = relu(conv(x_n, W_unique)),  s_n = relu(conv(x_n, W_shared)),  a_n = (u_n - s_n) + sum_m s_m,
// then score = softmax over the views of a_n per (voxel, channel) and out = sum_n score_n * x_n.  The two-kernel
// path (conv_ring.cu 8 -> 16 per view + k_attention_raw) writes and re-reads N * V * 16 fp16 logits (335 MB at cfg2
// against 252 MB of algorithmic traffic).  Here a CTA convolves ALL views of its tile column in the same plane
// step - the pipeline of conv_ring.cu (halo-plane ring in shared memory, in-plane taps as shifted UMMA descriptors,
// the three z taps side by side in N) with one ring plane and one accumulator ring PER VIEW:
//
//   ring slot    : [view][18 y][10 x][8 channels] 16-bit of one input z plane (no-swizzle K-major core matrices)
//   accumulators : TMEM columns [view][G groups][16 = u | s], one group per output plane; input plane i adds to the
//                  groups of the output planes i-2, i-1, i with B = [w_dz2 | w_dz1 | w_dz0] (N = 48; a run that
//                  wraps around the ring of G groups is issued as two MMAs)
//   epilogue     : a thread owns one voxel: 16 logits per view from TMEM, ReLU, softmax over the views in the order
//                  of k_attention_raw (net_fp32.cu), the views' centre voxels from global memory (L2: the producers
//                  fetched the same lines a few planes earlier), one 32-byte fp32 result per voxel
//   warps 0-3 producers (cp.async, zero fill = 'SAME' padding) | warp 4 MMA issuer | warps 5-8 epilogue
//
// DRAM traffic: the N views once (x 1.4 halo, mostly L2) + the fp32 result.
#include "ring_common.cuh"
#include "conv_ring.cuh"
#include <cstring>

namespace {

constexpr int AR_TY = 16, AR_TX = 8, AR_HH = AR_TY + 2, AR_WW = AR_TX + 2;
constexpr int AR_NVOX = AR_HH * AR_WW;              // 180 voxels of one halo plane
constexpr int AR_PLANE = AR_NVOX * 16 + 16;         // one view's plane (+16 B: bank skew between the views)
constexpr int AR_PRODUCERS = 128;
constexpr int AR_THREADS = 288;
constexpr int AR_CP = 16;                           // columns per (view, output plane): [u 8 | s 8]
constexpr int AR_NSTEPS = 5;                        // tap pairs (0,1) (2,3) (4,5) (6,7) (7*,8), conv_ring.cu
constexpr int AR_NROWS = 3 * AR_CP;                 // rows of one weight step image [w_dz2 | w_dz1 | w_dz0]
constexpr int AR_STEP_BYTES = 2 * AR_NROWS * 16;
constexpr int AR_MAXR = 16, AR_MAXG = 8, AR_MAXV = 8;

struct AttnParams {
    const void* x[AR_MAXV];
    int NV;
    int B, D, H, W;
    uint32_t fmt;
    int f16;            // views are fp16 (else bf16)
    int nXT, nYT;
    int nring, pf;
    int wbytes;
    long long total;    // tile columns * D
};

struct AUnit {
    int b, x0, y0, z0, zlen;
};

struct AUnitIter {
    RingSpan span;
    __device__ __forceinline__ explicit AUnitIter(const AttnParams& p) : span(p.total) {}
    __device__ __forceinline__ bool next(const AttnParams& p, AUnit& r) {
        long long t;
        if (!span.next(p.D, t, r.z0, r.zlen)) return false;
        r.x0 = (int)(t % p.nXT) * AR_TX;
        t /= p.nXT;
        r.y0 = (int)(t % p.nYT) * AR_TY;
        r.b = (int)(t / p.nYT);
        return true;
    }
};

__device__ __forceinline__ int aunit_ibeg(const AUnit& u) { return u.z0 == 0 ? 1 : 0; }
__device__ __forceinline__ int aunit_iend(const AttnParams& p, const AUnit& u) {
    return (u.z0 + u.zlen == p.D) ? u.zlen : u.zlen + 1;
}

// softmax over <= 8 views: arguments are <= 0 (max subtracted), a flushed-to-zero tail and 1-2 ulp are far below the
// 16-bit operands' rounding; exp2f() / IEEE division cost 6-8 instructions each, 40 of them per voxel
__device__ __forceinline__ float ex2_approx(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ float rcp_approx(float x) {
    float y;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

template <bool F16>
__device__ __forceinline__ void unpack8(const uint4& u, float* f) {
    const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        if (F16) {
            const float2 t = __half22float2(*reinterpret_cast<const __half2*>(&w[k]));
            f[2 * k] = t.x; f[2 * k + 1] = t.y;
        } else {
            f[2 * k] = __uint_as_float(w[k] << 16);
            f[2 * k + 1] = __uint_as_float(w[k] & 0xffff0000u);
        }
    }
}

// NMAX: views the kernel is built for (TMEM columns, ring slot size); p.NV <= NMAX of them are live
template <int NMAX, int G, int MINB, bool F16>
__global__ void __launch_bounds__(AR_THREADS, MINB)
k_attention_ring(const __grid_constant__ AttnParams p, const uint8_t* __restrict__ wimg, float* __restrict__ out) {
    constexpr int SLOT_BYTES = (NMAX * AR_PLANE + 127) / 128 * 128;
    constexpr uint32_t VIEW_COLS = (uint32_t)G * AR_CP;
    constexpr uint32_t TMEM_COLS = (uint32_t)NMAX * VIEW_COLS;
    static_assert(TMEM_COLS == 128 || TMEM_COLS == 256 || TMEM_COLS == 512, "TMEM columns: power of two");

    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>(((uintptr_t)smem_raw + 127) & ~(uintptr_t)127);
    uint8_t* wsm = smem;
    uint8_t* ring = smem + ((p.wbytes + 127) & ~127);
    uint64_t* bars = reinterpret_cast<uint64_t*>(ring + (size_t)p.nring * SLOT_BYTES);
    uint64_t* full = bars;
    uint64_t* empty = bars + p.nring;
    uint64_t* tfull = bars + 2 * p.nring;
    uint64_t* tempty = tfull + AR_MAXG;
    uint64_t* wbar = tempty + AR_MAXG;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(wbar + 1);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int R = p.nring;
    const int NV = p.NV;
    if (threadIdx.x == 0) {
        for (int s = 0; s < R; ++s) {
            mbar_init(&full[s], AR_PRODUCERS / 32);
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
                     "r"(TMEM_COLS)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    if (warp >= 5) {
        const uint32_t taddr = tmem_base + ((uint32_t)((warp & 3) * 32) << 16);
        for (uint32_t c = 0; c < TMEM_COLS; c += 8) tc_st8_zero(taddr + c);
        tc_wait_st();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();

    if (warp < 4) {
        // ===================== producers =====================
        const int ptid = threadIdx.x;
        if (ptid == 0) {
            mbar_expect_tx(wbar, (uint32_t)p.wbytes);
            bulk_copy_g2s(wsm, wimg, (uint32_t)p.wbytes, wbar);
        }
        constexpr int NITEM = (NMAX * AR_NVOX + AR_PRODUCERS - 1) / AR_PRODUCERS;
        const int PF = p.pf;
        uint32_t slot = 0, sphase = 0, pslot = 0, pending = 0;
        const uint32_t ring_u32 = smem_u32(ring);
        auto publish = [&](int keep) {
            if (keep >= 3) asm volatile("cp.async.wait_group 3;" ::: "memory");
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
        const size_t zstride_in = (size_t)p.H * p.W * 8;
        AUnitIter units(p);
        AUnit un;
        while (units.next(p, un)) {
            const int ibeg = aunit_ibeg(un), iend = aunit_iend(p, un);
            int goff[NITEM];       // element offset inside a z plane, -1 = zero fill, -2 = no item
#pragma unroll
            for (int k = 0; k < NITEM; ++k) {
                const int j = ptid + k * AR_PRODUCERS;
                const int v = j / AR_NVOX, vox = j - v * AR_NVOX;
                const int vy = vox / AR_WW, vx = vox - vy * AR_WW;
                const int gy = un.y0 - 1 + vy, gx = un.x0 - 1 + vx;
                const bool ok = gy >= 0 && gy < p.H && gx >= 0 && gx < p.W;
                goff[k] = (v >= NV) ? -2 : (ok ? (gy * p.W + gx) * 8 : -1);
            }
            size_t zoff = ((size_t)un.b * p.D + (un.z0 - 1 + ibeg)) * zstride_in;
            for (int i = ibeg; i <= iend; ++i, zoff += zstride_in) {
                mbar_wait(&empty[slot], sphase ^ 1);
                const uint32_t dst0 = ring_u32 + slot * (uint32_t)SLOT_BYTES;
#pragma unroll
                for (int k = 0; k < NITEM; ++k) {
                    if (goff[k] != -2) {
                        const int j = ptid + k * AR_PRODUCERS;
                        const int v = j / AR_NVOX, vox = j - v * AR_NVOX;
                        const uint32_t soff = (uint32_t)(v * AR_PLANE + vox * 16);
                        const bool ok = goff[k] >= 0;
                        const uint16_t* base = reinterpret_cast<const uint16_t*>(p.x[v]);
                        const uint16_t* src = ok ? base + zoff + goff[k] : base;
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
        if (elect_one()) {
            mbar_wait(wbar, 0);
            tc_fence_after();
            constexpr uint32_t A_HI = (uint32_t)((AR_WW * 16) >> 4) | (1u << 14);          // SBO = next y row
            constexpr uint32_t B_HI = (uint32_t)(128 >> 4) | (1u << 14);                    // SBO = next 8 rows
            const uint32_t FAST_IDESC = ring_idesc(3 * AR_CP) | p.fmt;
            const uint32_t a_lo_ring = smem_u32(ring) >> 4;
            const uint32_t b_lo0 = (smem_u32(wsm) >> 4) | ((uint32_t)((AR_NROWS * 16) >> 4) << 16);
            auto issue_plane = [&](uint32_t dcol, uint32_t a_lo0, uint32_t b_lo, uint32_t idesc) {
#pragma unroll
                for (int s = 0; s < AR_NSTEPS; ++s) {
                    const int ta = (s < 4) ? 2 * s : 7, tb = (s < 4) ? 2 * s + 1 : 8;
                    const uint32_t offa = (uint32_t)(((ta / 3) * AR_WW + (ta % 3)) * 16);
                    const uint32_t offb = (uint32_t)(((tb / 3) * AR_WW + (tb % 3)) * 16);
                    const uint32_t aoff = (offa >> 4) | (((offb - offa) >> 4) << 16);
                    tc_mma_lohi1(dcol, a_lo0 + aoff, A_HI, b_lo + ((uint32_t)(s * AR_STEP_BYTES) >> 4), B_HI, idesc);
                }
            };
            uint32_t slot = 0, sphase = 0;
            uint32_t gq = 0, gphase = 0;
            AUnitIter units(p);
            AUnit un;
            while (units.next(p, un)) {
                const int ibeg = aunit_ibeg(un), iend = aunit_iend(p, un);
                uint32_t gw = gq, gwphase = gphase;
                int twaited = -1;
                uint32_t glo = gq;
                uint32_t gdone = gq;
                int tdone = 0;
                for (int i = ibeg; i <= iend; ++i) {
                    const int tlo = max(0, i - 2), thi = min(un.zlen - 1, i);
                    while (twaited < thi) {
                        mbar_wait(&tempty[gw], gwphase ^ 1);
                        ++twaited;
                        if (++gw == (uint32_t)G) { gw = 0; gwphase ^= 1; }
                    }
                    mbar_wait(&full[slot], sphase);
                    tc_fence_after();
                    const uint32_t a_slot = a_lo_ring + slot * (uint32_t)(SLOT_BYTES >> 4);
                    const int len = thi - tlo + 1, f = i - tlo;
                    const int len1 = min(len, G - (int)glo), len2 = len - len1;
                    for (int v = 0; v < NV; ++v) {
                        const uint32_t a_lo0 = a_slot + (uint32_t)v * (uint32_t)(AR_PLANE >> 4);
                        const uint32_t dview = tmem_base + (uint32_t)v * VIEW_COLS;
                        if (len == 3 && len2 == 0) {
                            issue_plane(dview + glo * (uint32_t)AR_CP, a_lo0, b_lo0, FAST_IDESC);
                        } else {
                            const uint32_t boff1 = (uint32_t)(2 - f) * (uint32_t)AR_CP * 16u;
                            issue_plane(dview + glo * (uint32_t)AR_CP, a_lo0, b_lo0 + (boff1 >> 4),
                                        ring_idesc(len1 * AR_CP) | p.fmt);
                            if (len2 > 0) {
                                const uint32_t boff2 = (uint32_t)(2 - (f - len1)) * (uint32_t)AR_CP * 16u;
                                issue_plane(dview, a_lo0, b_lo0 + (boff2 >> 4), ring_idesc(len2 * AR_CP) | p.fmt);
                            }
                        }
                    }
                    tc_commit(&empty[slot]);
                    if (++slot == (uint32_t)R) { slot = 0; sphase ^= 1; }
                    if (i >= 2 && ++glo == (uint32_t)G) glo = 0;
                    const int tlast = (i == iend) ? un.zlen - 1 : i - 2;
                    while (tdone <= tlast) {
                        tc_commit(&tfull[gdone]);
                        ++tdone;
                        if (++gdone == (uint32_t)G) gdone = 0;
                    }
                }
                gq = gw; gphase = gwphase;
            }
        }
        __syncwarp();
    } else {
        // ===================== epilogue (4 warps = 128 TMEM lanes, one voxel per thread) =====================
        const int g = warp & 3;
        const int row = g * 32 + lane;
        const int ty = row >> 3, tx = row & 7;
        uint32_t grp = 0, gphase = 0;
        AUnitIter units(p);
        AUnit un;
        while (units.next(p, un)) {
            const int y = un.y0 + ty, x = un.x0 + tx;
            const bool ok = y < p.H && x < p.W;
            const size_t zstride = (size_t)p.H * p.W * 8;
            size_t voff = ((((size_t)un.b * p.D + un.z0) * p.H + (ok ? y : 0)) * p.W + (ok ? x : 0)) * 8;
            for (int t = 0; t < un.zlen; ++t, voff += zstride) {
                // the views' centre voxels: issued before the wait, consumed after the softmax
                uint4 xr[NMAX];
#pragma unroll
                for (int n = 0; n < NMAX; ++n)
                    if (n < NV && ok) xr[n] = __ldg(reinterpret_cast<const uint4*>(reinterpret_cast<const uint16_t*>(p.x[n]) + voff));
                mbar_wait(&tfull[grp], gphase);
                tc_fence_after();
                const uint32_t taddr = tmem_base + ((uint32_t)(g * 32) << 16) + grp * (uint32_t)AR_CP;
                uint64_t* const tempty_bar = &tempty[grp];
                if (++grp == (uint32_t)G) { grp = 0; gphase ^= 1; }
                // l_n = relu(u_n) - relu(s_n): the "+ sum_m s_m" of network.py:344 is the same for every view and cancels in
                // the softmax over views (as in the sharded form, pipeline.aggregate), so it is not formed at all
                float a[NMAX][8];
#pragma unroll
                for (int n = 0; n < NMAX; ++n) {
                    if (n < NV) {
                        // one view per TMEM round trip: two at a time costs the 4-view build (96 registers at two CTAs
                        // per SM) 80 bytes of spills and 14 us
                        float us[16];
                        tc_ld16(taddr + (uint32_t)n * VIEW_COLS, us);
                        tc_wait_ld();
#pragma unroll
                        for (int q = 0; q < 8; ++q) a[n][q] = fmaxf(us[q], 0.f) - fmaxf(us[8 + q], 0.f);
                        tc_st8_zero(taddr + (uint32_t)n * VIEW_COLS);
                        tc_st8_zero(taddr + (uint32_t)n * VIEW_COLS + 8);
                    }
                }
                tc_wait_st();
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(tempty_bar);
                if (!ok) continue;
                constexpr float LOG2E = 1.4426950408889634f;
                float mneg[8], den[8], res[8];
#pragma unroll
                for (int q = 0; q < 8; ++q) {
                    float mm = a[0][q];
#pragma unroll
                    for (int n = 1; n < NMAX; ++n)
                        if (n < NV) mm = fmaxf(mm, a[n][q]);
                    mneg[q] = -mm * LOG2E;
                    den[q] = 0.f;
                    res[q] = 0.f;
                }
#pragma unroll
                for (int n = 0; n < NMAX; ++n)
                    if (n < NV) {
                        float xx[8];
                        unpack8<F16>(xr[n], xx);
#pragma unroll
                        for (int q = 0; q < 8; ++q) {
                            const float e = ex2_approx(fmaf(a[n][q], LOG2E, mneg[q]));      // exp(l_n - max)
                            den[q] += e;
                            res[q] = fmaf(e, xx[q], res[q]);
                        }
                    }
#pragma unroll
                for (int q = 0; q < 8; ++q) res[q] *= rcp_approx(den[q]);
                float4* o = reinterpret_cast<float4*>(out + voff);
                o[0] = make_float4(res[0], res[1], res[2], res[3]);
                o[1] = make_float4(res[4], res[5], res[6], res[7]);
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 4) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS)
                     : "memory");
    }
}

template <int NMAX, int G, int MINB, bool F16>
int launch_attn(const AttnParams& p, const uint8_t* wimg, float* out, size_t smem, int grid, cudaStream_t st) {
    if (const int rc = atvs_max_dynamic_smem<k_attention_ring<NMAX, G, MINB, F16>>()) return rc;
    k_attention_ring<NMAX, G, MINB, F16><<<grid, AR_THREADS, smem, st>>>(p, wimg, out);
    ATVS_LAUNCH_CHECK();
    return 0;
}

}  // namespace

bool attn_ring_applicable(int n_views, int D, int H, int W) {
    return n_views >= 2 && n_views <= AR_MAXV && D >= 3 && H >= 8 && W >= 8;
}

// wimg: the halo-ring weight image of the 8 -> 16 convolution [W_unique | W_shared] (ring_pack(…, 8, 16, …))
int attn_ring(const void* const* views, int n_views, int dtype, const void* wimg, int B, int D, int H, int W, float* out,
              cudaStream_t st) {
    AttnParams p;
    memset(&p, 0, sizeof(p));
    for (int n = 0; n < n_views; ++n) p.x[n] = views[n];
    p.NV = n_views;
    p.B = B; p.D = D; p.H = H; p.W = W;
    p.fmt = tc_fmt_bits(dtype);
    p.f16 = dtype == ATVS_F16;
    p.nXT = (W + AR_TX - 1) / AR_TX;
    p.nYT = (H + AR_TY - 1) / AR_TY;
    p.wbytes = AR_NSTEPS * AR_STEP_BYTES;
    p.total = (long long)B * p.nXT * p.nYT * D;
    const int nmax = n_views <= 2 ? 2 : (n_views <= 4 ? 4 : 8);
    const int minb = nmax <= 4 ? 2 : 1;
    const size_t slot = ((size_t)nmax * AR_PLANE + 127) / 128 * 128;
    const size_t fixed = 128 + (size_t)((p.wbytes + 127) & ~127) + (2 * AR_MAXR + 2 * AR_MAXG + 1) * 8 + 16;
    const size_t budget = (minb == 2 ? 110 : 220) * 1024;
    int nring = (int)((budget - fixed) / slot);
    if (nring > 8) nring = 8;
    if (nring < 2) {
        atvs_set_error("atvs_attention_fused: ring does not fit");
        return ATVS_E_UNSUP;
    }
    p.nring = nring;
    p.pf = nring - 1 < 4 ? nring - 1 : 4;
    const size_t smem = fixed + (size_t)nring * slot;
    const int sms = atvs_num_sms();
    const int grid = ring_balanced_grid(p.total, (long long)sms * minb, 12, 40);
    const uint8_t* wi = (const uint8_t*)wimg;
#define AT_CASE(NM, GG, MB)                                                                                  \
    return p.f16 ? launch_attn<NM, GG, MB, true>(p, wi, out, smem, grid, st)                                 \
                 : launch_attn<NM, GG, MB, false>(p, wi, out, smem, grid, st)
    if (nmax == 2) { AT_CASE(2, 8, 2); }
    if (nmax == 4) { AT_CASE(4, 4, 2); }
    AT_CASE(8, 4, 1);
#undef AT_CASE
}
