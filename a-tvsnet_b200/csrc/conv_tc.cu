// conv_tc.cu - 3-D convolution / transposed convolution as an implicit GEMM on the Blackwell
// 5th-generation tensor cores (tcgen05.mma, accumulators in TMEM, operands staged by TMA),
// bf16 operands, fp32 accumulation.  Replaces tf.layers.conv3d / conv3d_transpose of
// network.py:173-215, 511-550 (cuDNN fp32 in the reference) for the cost-regularisation
// network and the attention convolutions.
//
// Formulation (one CTA = one persistent worker, 6 warps):
//   GEMM M = 128 output voxels of a (TD,TH,TW) brick, N = Cout (padded to 16/32/64),
//   K = Cin per filter tap.  For every tap ONE TMA box load of the (shifted) input brick
//   [TD][TH][TW][Cin] is a K-major A tile (row = voxel, 2*Cin bytes, swizzle = row bytes);
//   TMA's out-of-bounds zero fill IS the 'SAME' zero padding.  Stride-2 convolutions read
//   through 8 parity-view tensor maps (in = 2j + off), transposed convolutions run one
//   launch per output parity class (conv_geom.cuh).  All taps' weights stay resident in
//   shared memory ([tap][N][Cin] K-major tiles loaded once per CTA by TMA).
//   warp 0: TMA producer | warp 1: TMEM allocator + single-thread MMA issuer |
//   warps 2-5: epilogue (tcgen05.ld -> raw fp32 store + per-channel sum / sum-of-squares for
//   the batch-statistics BN), double-buffered TMEM accumulators.
//   Cin = 8 (16-byte rows): two taps form one K=16 step (no-swizzle core-matrix layout, the
//   second tap's tile is the K-adjacent core matrix, LBO = tile size).
#include "tc_ptx.cuh"
#include "conv_geom.cuh"
#include "conv_ring.cuh"
#include "conv_deconv.cuh"
#include <cstring>

namespace {

constexpr int TC_MAX_TAPS = 48;      // 27 for a 3-D kernel; 2-D: 9 taps x up to 5 chunks of 64 input channels
constexpr int TC_THREADS = 192;

struct TcTap {
    int map, ox, oy, oz;
};

struct TcParams {
    int ntaps;                 // padded to a multiple of taps-per-stage
    TcTap taps[TC_MAX_TAPS];
    int B, Dj, Hj, Wj;         // iteration space (tile origins live here)
    int Do, Ho, Wo;            // full output extent
    int os;                    // out = j*os + parity
    int ncls;                  // parity classes merged in this launch (1 for convolutions, 8 for deconv)
    int cls_tap0[9];           // class c uses taps [cls_tap0[c], cls_tap0[c+1])
    int cls_par[8][3];         // output parity (z, y, x) of class c
    int ltd, lth, ltw;         // log2 of the brick dims (TD*TH*TW == 128)
    int nTD, nTH, nTW;
    int Cout, coff, ncols;     // real channel count, slab offset, real columns in this slab
    int raw16;                 // raw output dtype: 0 fp32, 1 saturated fp16
    uint32_t fmt;              // operand format bits of the instruction descriptor (tc_fmt_bits)
    unsigned long long* sat;   // saturation counter of the fp16 raw stores (atvs_sat_ptr)
    const float* chan_bias;    // per-channel bias (Cout) added in the epilogue, or NULL (2-D layers of the FEM)
    int relu;                  // ReLU in the epilogue (after the bias)
    int nstages;
    long long ntiles;
};

struct alignas(64) TcMaps {
    CUtensorMap a[8];
    CUtensorMap w;
};

template <int CIN>
struct TcCfg {
    static constexpr int TPS = (CIN == 8) ? 2 : 1;              // taps per pipeline stage
    static constexpr int KSTEPS = (CIN >= 16) ? CIN / 16 : 1;   // UMMA K=16 steps per stage
    static constexpr int TILE_BYTES = 128 * CIN * 2;
    static constexpr int STAGE_BYTES = TILE_BYTES * TPS;
    // UMMA layout_type: 0 none, 2 = 128B, 4 = 64B, 6 = 32B
    static constexpr uint32_t LAYOUT = (CIN == 64) ? 2u : (CIN == 32) ? 4u : (CIN == 16) ? 6u : 0u;
    static constexpr uint32_t SBO = (CIN == 8) ? 128u : (uint32_t)(8 * CIN * 2);
};

template <int CIN, int NPAD>
__global__ void __launch_bounds__(TC_THREADS, 1)
k_conv3d_tc(const __grid_constant__ TcMaps tm, const __grid_constant__ TcParams p, float* __restrict__ out,
            double* __restrict__ stats, const float* __restrict__ bias) {
    using Cfg = TcCfg<CIN>;
    constexpr int WTAP_BYTES = NPAD * CIN * 2;
    constexpr uint32_t TMEM_COLS = (2 * NPAD < 32) ? 32u : (uint32_t)(2 * NPAD);
    const uint32_t IDESC = (1u << 4) | ((uint32_t)(NPAD >> 3) << 17) | ((128u >> 4) << 24) | p.fmt;

    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    uint8_t* wsm = smem;
    const int wbytes = p.ntaps * WTAP_BYTES;
    uint8_t* asmem = smem + ((wbytes + 1023) & ~1023);
    uint64_t* bars = reinterpret_cast<uint64_t*>(asmem + (size_t)p.nstages * Cfg::STAGE_BYTES);
    uint64_t* full = bars;
    uint64_t* empty = bars + p.nstages;
    uint64_t* tfull = bars + 2 * p.nstages;
    uint64_t* tempty = tfull + 2;
    uint64_t* wbar = tempty + 2;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(wbar + 1);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) {
        for (int s = 0; s < p.nstages; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], 1);
        }
        mbar_init(&tfull[0], 1);
        mbar_init(&tfull[1], 1);
        mbar_init(&tempty[0], 4);
        mbar_init(&tempty[1], 4);
        mbar_init(wbar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                     "r"(TMEM_COLS)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    const int tiles_per_b = p.nTD * p.nTH * p.nTW;
    const long long nwork = p.ntiles * p.ncls;      // work item = (class, tile), class-major

    if (warp == 0) {
        // ===================== TMA producer (converged warp, elected lane issues) =====================
        {
            const uint32_t leader = elect_one();
            mbar_expect_tx_leader(wbar, (uint32_t)wbytes, leader);
            for (int t = 0; t < p.ntaps; ++t)
                tma_load_2d_leader(wsm + (size_t)t * WTAP_BYTES, &tm.w, 0, t * NPAD, wbar, leader);
            int stage = 0;
            uint32_t phase = 0;
            for (long long wk = blockIdx.x; wk < nwork; wk += gridDim.x) {
                const int cls = (int)(wk / p.ntiles);
                const long long tile = wk % p.ntiles;
                const int t0 = p.cls_tap0[cls], nsteps = (p.cls_tap0[cls + 1] - t0) / Cfg::TPS;
                const int b = (int)(tile / tiles_per_b);
                int r = (int)(tile % tiles_per_b);
                const int jx0 = (r % p.nTW) << p.ltw;
                r /= p.nTW;
                const int jy0 = (r % p.nTH) << p.lth;
                const int jz0 = (r / p.nTH) << p.ltd;
                for (int s = 0; s < nsteps; ++s) {
                    mbar_wait(&empty[stage], phase ^ 1);
                    mbar_expect_tx_leader(&full[stage], (uint32_t)Cfg::STAGE_BYTES, leader);
                    uint8_t* dst = asmem + (size_t)stage * Cfg::STAGE_BYTES;
#pragma unroll
                    for (int q = 0; q < Cfg::TPS; ++q) {
                        const TcTap& tp = p.taps[t0 + s * Cfg::TPS + q];
                        tma_load_5d_leader(dst + q * Cfg::TILE_BYTES, &tm.a[tp.map], 0, jx0 + tp.ox, jy0 + tp.oy,
                                           jz0 + tp.oz, b, &full[stage], leader);
                    }
                    if (++stage == p.nstages) {
                        stage = 0;
                        phase ^= 1;
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ===================== MMA issuer (converged warp, elected lane issues) =====================
        {
            const uint32_t leader = elect_one();
            mbar_wait(wbar, 0);
            tc_fence_after();
            const uint32_t a_lbo = (CIN == 8) ? (uint32_t)Cfg::TILE_BYTES : 16u;
            const uint32_t b_lbo = (CIN == 8) ? (uint32_t)(NPAD * 16) : 16u;
            const uint64_t wdesc0 = make_desc(smem_u32(wsm), b_lbo, Cfg::SBO, Cfg::LAYOUT);
            int stage = 0;
            uint32_t phase = 0;
            long long it = 0;
            for (long long wk = blockIdx.x; wk < nwork; wk += gridDim.x, ++it) {
                const int cls = (int)(wk / p.ntiles);
                const int t0 = p.cls_tap0[cls], nsteps = (p.cls_tap0[cls + 1] - t0) / Cfg::TPS;
                const int acc = (int)(it & 1);
                mbar_wait(&tempty[acc], (uint32_t)(((it >> 1) & 1) ^ 1));
                tc_fence_after();
                const uint32_t dcol = tmem_base + (uint32_t)(acc * NPAD);
                for (int s = 0; s < nsteps; ++s) {
                    mbar_wait(&full[stage], phase);
                    tc_fence_after();
                    const uint64_t ad0 = make_desc(smem_u32(asmem + (size_t)stage * Cfg::STAGE_BYTES), a_lbo, Cfg::SBO, Cfg::LAYOUT);
                    const uint64_t bd0 = desc_advance(wdesc0, (uint32_t)((t0 + s * Cfg::TPS) * WTAP_BYTES));
#pragma unroll
                    for (int ks = 0; ks < Cfg::KSTEPS; ++ks) {
                        const uint64_t ad = desc_advance(ad0, ks * 32), bd = desc_advance(bd0, ks * 32);
                        if (ks == 0 && s == 0) tc_mma_bf16_first(dcol, ad, bd, IDESC, leader);
                        else tc_mma_bf16_acc(dcol, ad, bd, IDESC, leader);
                    }
                    tc_commit_leader(&empty[stage], leader);
                    if (++stage == p.nstages) {
                        stage = 0;
                        phase ^= 1;
                    }
                }
                tc_commit_leader(&tfull[acc], leader);
            }
        }
    } else {
        // ===================== epilogue (4 warps = 128 TMEM lanes) =====================
        const int g = warp & 3;
        const int row = g * 32 + lane;
        const int tw = row & ((1 << p.ltw) - 1);
        const int th = (row >> p.ltw) & ((1 << p.lth) - 1);
        const int td = row >> (p.ltw + p.lth);
        constexpr int NRED = 2 * NPAD;              // per-thread running moments
        float run[NRED];
#pragma unroll
        for (int i = 0; i < NRED; ++i) run[i] = 0.f;
        long long it = 0;
        for (long long wk = blockIdx.x; wk < nwork; wk += gridDim.x, ++it) {
            const int cls = (int)(wk / p.ntiles);
            const long long tile = wk % p.ntiles;
            const int pz = p.cls_par[cls][0], py = p.cls_par[cls][1], px = p.cls_par[cls][2];
            const int acc = (int)(it & 1);
            const int b = (int)(tile / tiles_per_b);
            int r = (int)(tile % tiles_per_b);
            const int jx = ((r % p.nTW) << p.ltw) + tw;
            r /= p.nTW;
            const int jy = ((r % p.nTH) << p.lth) + th;
            const int jz = ((r / p.nTH) << p.ltd) + td;
            const bool valid = jx < p.Wj && jy < p.Hj && jz < p.Dj;
            mbar_wait(&tfull[acc], (uint32_t)((it >> 1) & 1));
            tc_fence_after();
            const uint32_t taddr = tmem_base + ((uint32_t)(g * 32) << 16) + (uint32_t)(acc * NPAD);
            const size_t o = valid ? ((((size_t)b * p.Do + (jz * p.os + pz)) * p.Ho + (jy * p.os + py)) * p.Wo +
                                      (jx * p.os + px)) * p.Cout + p.coff : 0;
            const float* brow = p.chan_bias != nullptr ? p.chan_bias + p.coff : nullptr;
            if (bias != nullptr && valid) {      // convolutions only (os == 1): plane classes first / interior / last
                const int zc = (jz == 0) ? 0 : (jz == p.Do - 1 ? 2 : 1);
                brow = bias + ((((size_t)b * 3 + zc) * p.Ho + jy) * p.Wo + jx) * p.Cout + p.coff;
            }
            epilogue_tile<NPAD>(taddr, &tempty[acc], lane, valid, out, o, p.ncols,
                                raw_vec_mode(out, p.ncols, p.Cout, p.coff), p.raw16, stats != nullptr, run, brow, p.sat,
                                p.relu != 0);
        }
        if (stats != nullptr) flush_stats<NPAD>(stats, run, lane, p.Cout, p.coff, p.ncols);
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
    }
}

// ------------------------------------------------------------------ weight packing
// packed image: for each class, for each (padded) tap, for each slab: [NPAD][Cin] bf16, K-major.
__global__ void k_pack_weights(const float* __restrict__ w, int Cin, int Cout, int transposed, int npad, int nslabs,
                               int ncls, int f16, unsigned short* __restrict__ out) {
    // one block per (class, slab, tap); taps follow make_conv_geom order
    const int tps = (Cin == 8) ? 2 : 1;
    int cls = 0, slab = 0, tap = 0, ntaps_pad = 0;
    size_t base = 0;
    {
        int blk = blockIdx.x;
        for (cls = 0; cls < ncls; ++cls) {
            const ConvGeom g = make_conv_geom(1, 2, 2, 2, Cin, Cout, 1, transposed, cls);
            const int nt = g.nt[0] * g.nt[1] * g.nt[2];
            ntaps_pad = (nt + tps - 1) / tps * tps;
            if (blk < ntaps_pad * nslabs) break;
            blk -= ntaps_pad * nslabs;
            base += (size_t)ntaps_pad * nslabs * npad * Cin;
        }
        if (cls == ncls) return;
        slab = blk / ntaps_pad;
        tap = blk % ntaps_pad;
    }
    const ConvGeom g = make_conv_geom(1, 2, 2, 2, Cin, Cout, 1, transposed, cls);
    const int nt = g.nt[0] * g.nt[1] * g.nt[2];
    int kidx = -1;
    if (tap < nt) {
        const int tx = tap % g.nt[2], ty = (tap / g.nt[2]) % g.nt[1], tz = tap / (g.nt[2] * g.nt[1]);
        kidx = (g.kidx[0][tz] * 3 + g.kidx[1][ty]) * 3 + g.kidx[2][tx];
    }
    unsigned short* o = out + base + ((size_t)slab * ntaps_pad + tap) * npad * Cin;
    for (int i = threadIdx.x; i < npad * Cin; i += blockDim.x) {
        const int n = i / Cin, k = i % Cin;
        const int co = slab * npad + n;
        float val = 0.f;
        if (kidx >= 0 && co < Cout)
            val = transposed ? w[((size_t)kidx * Cout + co) * Cin + k] : w[((size_t)kidx * Cin + k) * Cout + co];
        o[i] = tc_cvt16(val, f16);
    }
}

// ------------------------------------------------------------------ host side
CUtensorMapSwizzle swizzle_for(int cin) {
    return cin == 64 ? CU_TENSOR_MAP_SWIZZLE_128B
         : cin == 32 ? CU_TENSOR_MAP_SWIZZLE_64B
         : cin == 16 ? CU_TENSOR_MAP_SWIZZLE_32B
                     : CU_TENSOR_MAP_SWIZZLE_NONE;
}

struct SlabPlan {
    int npad, nslabs;
};

// pick the N tile: the smallest of {16,32,64} covering Cout whose resident weights fit
SlabPlan plan_slabs(int Cin, int Cout, int max_taps) {
    int npad = Cout <= 16 ? 16 : Cout <= 32 ? 32 : 64;
    const int tps = (Cin == 8) ? 2 : 1;
    const int tp = (max_taps + tps - 1) / tps * tps;
    while (npad > 16 && (size_t)tp * npad * Cin * 2 > 120 * 1024) npad >>= 1;
    return SlabPlan{npad, (Cout + npad - 1) / npad};
}

int ntaps_padded(int Cin, int transposed, int cls) {
    const ConvGeom g = make_conv_geom(1, 2, 2, 2, Cin, 16, 1, transposed, cls);
    const int nt = g.nt[0] * g.nt[1] * g.nt[2];
    const int tps = (Cin == 8) ? 2 : 1;
    return (nt + tps - 1) / tps * tps;
}

template <int CIN, int NPAD>
int launch_tc(const TcMaps& maps, const TcParams& p, float* out, double* stats, const float* bias, size_t smem,
              int grid, cudaStream_t st) {
    if (const int rc = atvs_max_dynamic_smem<k_conv3d_tc<CIN, NPAD>>()) return rc;
    k_conv3d_tc<CIN, NPAD><<<grid, TC_THREADS, smem, st>>>(maps, p, out, stats, bias);
    ATVS_LAUNCH_CHECK();
    return 0;
}

}  // namespace

extern "C" size_t atvs_packed_weight_bytes(int Cin, int Cout, int transposed) {
    if (!(Cin == 8 || Cin == 16 || Cin == 32 || Cin == 64) || Cout < 1 || Cout > 64) return 0;
    const SlabPlan sp = plan_slabs(Cin, Cout, transposed ? 8 : 27);
    size_t elems = 0;
    const int ncls = transposed ? 8 : 1;
    for (int c = 0; c < ncls; ++c) elems += (size_t)ntaps_padded(Cin, transposed, c) * sp.nslabs * sp.npad * Cin;
    size_t bytes = (elems * 2 + 255) & ~(size_t)255;          // per-tap TMA image
    if (!transposed) bytes += ring_weight_bytes(Cin, Cout) + ring_s2_weight_bytes(Cin, Cout);   // halo-ring images (stride 1 | 2)
    else {
        if (deconv_fused_applicable(Cin, Cout)) bytes += (deconv_fused_weight_bytes(Cin, Cout) + 255) & ~(size_t)255;   // 8-class deconv image
        if (deconv_ring_supported(Cin, Cout)) bytes += deconv_ring_weight_bytes(Cin, Cout);     // plane-ring deconv image
    }
    return bytes;
}

static size_t tap_image_bytes(int Cin, int Cout, int transposed) {
    const SlabPlan sp = plan_slabs(Cin, Cout, transposed ? 8 : 27);
    size_t elems = 0;
    const int ncls = transposed ? 8 : 1;
    for (int c = 0; c < ncls; ++c) elems += (size_t)ntaps_padded(Cin, transposed, c) * sp.nslabs * sp.npad * Cin;
    return (elems * 2 + 255) & ~(size_t)255;
}

// CTAs of a per-tap launch.  Every CTA pays a fixed cost (TMEM allocation, all taps' weights into shared memory, pipeline
// fill) worth several tiles; a launch that owns the GPU wants one CTA per SM, but in a step whose passes share the SMs
// (atvs_set_concurrency > 1) fewer CTAs with more tiles each spend less SM time on the same work.
// Tiles per CTA when the SMs are shared, whole cfg2 step: 5.51 (1) 5.47 (2) 5.45 (4) 5.45 (6) 5.47 (8) 5.71 ms (12).
constexpr int TC_SHARED_MINTILES = 4;
static int tc_grid(long long nwork, int sms) {
    const int mint = atvs_concurrency() > 1 ? TC_SHARED_MINTILES : 1;
    long long g = nwork / mint;
    if (g < 1) g = 1;
    if (g > sms) g = sms;
    if (g > nwork) g = nwork;
    return (int)g;
}

extern "C" int atvs_pack_conv_weights_tc(const float* kernel, int Cin, int Cout, int transposed, int dtype, void* wpacked,
                                         atvs_stream_t stream) {
    ATVS_CHECK_ARG(kernel && wpacked, ATVS_E_NULL, "atvs_pack_conv_weights_tc: NULL pointer");
    ATVS_CHECK_ARG(dtype == ATVS_BF16 || dtype == ATVS_F16, ATVS_E_DTYPE, "atvs_pack_conv_weights_tc: dtype %d (ATVS_BF16 | ATVS_F16)", dtype);
    ATVS_CHECK_ARG(Cin == 8 || Cin == 16 || Cin == 32 || Cin == 64, ATVS_E_UNSUP,
                   "atvs_pack_conv_weights_tc: Cin=%d (8, 16, 32 or 64)", Cin);
    ATVS_CHECK_ARG(Cout >= 1 && Cout <= 64, ATVS_E_UNSUP, "atvs_pack_conv_weights_tc: Cout=%d (1..64)", Cout);
    const SlabPlan sp = plan_slabs(Cin, Cout, transposed ? 8 : 27);
    const int ncls = transposed ? 8 : 1;
    int blocks = 0;
    for (int c = 0; c < ncls; ++c) blocks += ntaps_padded(Cin, transposed, c) * sp.nslabs;
    k_pack_weights<<<blocks, 128, 0, (cudaStream_t)stream>>>(kernel, Cin, Cout, transposed, sp.npad, sp.nslabs, ncls,
                                                            dtype == ATVS_F16, (unsigned short*)wpacked);
    ATVS_LAUNCH_CHECK();
    if (!transposed) {
        int rc = ring_pack(kernel, Cin, Cout, dtype, (char*)wpacked + tap_image_bytes(Cin, Cout, 0), (cudaStream_t)stream);
        if (rc == 0 && ring_s2_supported(Cin, Cout))
            rc = ring_s2_pack(kernel, Cin, Cout, dtype,
                              (char*)wpacked + tap_image_bytes(Cin, Cout, 0) + ring_weight_bytes(Cin, Cout), (cudaStream_t)stream);
        return rc;
    }
    int rc = 0;
    size_t off = tap_image_bytes(Cin, Cout, 1);
    if (deconv_fused_applicable(Cin, Cout)) {
        rc = deconv_fused_pack(kernel, Cin, Cout, dtype, (char*)wpacked + off, (cudaStream_t)stream);
        off += (deconv_fused_weight_bytes(Cin, Cout) + 255) & ~(size_t)255;
    }
    if (rc == 0 && deconv_ring_supported(Cin, Cout))
        rc = deconv_ring_pack(kernel, Cin, Cout, dtype, (char*)wpacked + off, (cudaStream_t)stream);
    return rc;
}

static int conv3d_tc_impl(const void* x16, int x_dtype, const void* wpacked, int B, int D, int H, int W, int Cin, int Cout,
                          int stride, int transposed, const float* plane_bias, void* raw_out_v, int raw_dtype,
                          double* stats, atvs_stream_t stream);

extern "C" int atvs_attention_fused(const void* const* x_views, int N, int x_dtype, const void* wpacked, int B, int D, int H,
                                    int W, int C, float* out, atvs_stream_t stream) {
    ATVS_CHECK_ARG(x_views && wpacked && out, ATVS_E_NULL, "atvs_attention_fused: NULL pointer");
    ATVS_CHECK_ARG(x_dtype == ATVS_BF16 || x_dtype == ATVS_F16, ATVS_E_DTYPE,
                   "atvs_attention_fused: x_dtype %d (ATVS_BF16 or ATVS_F16)", x_dtype);
    ATVS_CHECK_ARG(C == 8, ATVS_E_UNSUP, "atvs_attention_fused: C=%d (8)", C);
    ATVS_CHECK_ARG(B > 0 && D > 0 && H > 0 && W > 0, ATVS_E_SHAPE, "atvs_attention_fused: bad shape");
    ATVS_CHECK_ARG(attn_ring_applicable(N, D, H, W), ATVS_E_UNSUP,
                   "atvs_attention_fused: N=%d (2..8 views), D=%d (>= 3), H=%d, W=%d (>= 8)", N, D, H, W);
    ATVS_CHECK_ARG((((uintptr_t)wpacked | (uintptr_t)out) & 15) == 0, ATVS_E_SHAPE,
                   "atvs_attention_fused: buffers must be 16-byte aligned");
    for (int n = 0; n < N; ++n)
        ATVS_CHECK_ARG(x_views[n] && ((uintptr_t)x_views[n] & 15) == 0, ATVS_E_NULL,
                       "atvs_attention_fused: view %d is NULL or not 16-byte aligned", n);
    return attn_ring(x_views, N, x_dtype, (const char*)wpacked + tap_image_bytes(8, 16, 0), B, D, H, W, out,
                     (cudaStream_t)stream);
}

extern "C" int atvs_conv3d_tc(const void* x16, int x_dtype, const void* wpacked, int B, int D, int H, int W, int Cin,
                              int Cout, int stride, int transposed, void* raw_out, int raw_dtype, double* stats,
                              atvs_stream_t stream) {
    return conv3d_tc_impl(x16, x_dtype, wpacked, B, D, H, W, Cin, Cout, stride, transposed, nullptr, raw_out, raw_dtype, stats,
                          stream);
}

extern "C" int atvs_conv3d_tc_bias(const void* x16, int x_dtype, const void* wpacked, int B, int D, int H, int W, int Cin,
                                   int Cout, int stride, const float* plane_bias, void* raw_out, int raw_dtype,
                                   double* stats, atvs_stream_t stream) {
    ATVS_CHECK_ARG(plane_bias, ATVS_E_NULL, "atvs_conv3d_tc_bias: plane_bias is NULL");
    ATVS_CHECK_ARG(((uintptr_t)plane_bias & 15) == 0, ATVS_E_SHAPE, "atvs_conv3d_tc_bias: plane_bias must be 16-byte aligned");
    ATVS_CHECK_ARG((D + stride - 1) / stride >= 2, ATVS_E_SHAPE, "atvs_conv3d_tc_bias: needs at least 2 output planes");
    return conv3d_tc_impl(x16, x_dtype, wpacked, B, D, H, W, Cin, Cout, stride, 0, plane_bias, raw_out, raw_dtype, stats, stream);
}

static int conv3d_tc_impl(const void* x_bf16, int x_dtype, const void* wpacked, int B, int D, int H, int W, int Cin, int Cout,
                          int stride, int transposed, const float* plane_bias, void* raw_out_v, int raw_dtype,
                          double* stats, atvs_stream_t stream) {
    ATVS_CHECK_ARG(x_dtype == ATVS_BF16 || x_dtype == ATVS_F16, ATVS_E_DTYPE,
                   "atvs_conv3d_tc: x_dtype %d (ATVS_BF16 or ATVS_F16)", x_dtype);
    float* raw_out = (float*)raw_out_v;        // element offsets are dtype independent; kernels re-type the base
    ATVS_CHECK_ARG(x_bf16 && wpacked && raw_out, ATVS_E_NULL, "atvs_conv3d_tc: NULL pointer");
    ATVS_CHECK_ARG(raw_dtype == ATVS_F32 || raw_dtype == ATVS_F16, ATVS_E_DTYPE,
                   "atvs_conv3d_tc: raw_dtype %d (ATVS_F32 or ATVS_F16)", raw_dtype);
    const int raw16 = raw_dtype == ATVS_F16;
    ATVS_CHECK_ARG(B > 0 && D > 0 && H > 0 && W > 0, ATVS_E_SHAPE, "atvs_conv3d_tc: bad shape");
    ATVS_CHECK_ARG(Cin == 8 || Cin == 16 || Cin == 32 || Cin == 64, ATVS_E_UNSUP,
                   "atvs_conv3d_tc: Cin=%d (8, 16, 32 or 64)", Cin);
    ATVS_CHECK_ARG(Cout >= 1 && Cout <= 64, ATVS_E_UNSUP, "atvs_conv3d_tc: Cout=%d (1..64)", Cout);
    ATVS_CHECK_ARG(transposed ? stride == 2 : (stride == 1 || stride == 2), ATVS_E_UNSUP,
                   "atvs_conv3d_tc: stride=%d transposed=%d", stride, transposed);
    ATVS_CHECK_ARG(transposed || stride == 1 || ((D | H | W) & 1) == 0, ATVS_E_DIV8,
                   "atvs_conv3d_tc: stride-2 convolution needs even D,H,W (got %d,%d,%d)", D, H, W);
    ATVS_CHECK_ARG(((uintptr_t)x_bf16 & 15) == 0 && ((uintptr_t)wpacked & 15) == 0 && ((uintptr_t)raw_out & 15) == 0,
                   ATVS_E_SHAPE, "atvs_conv3d_tc: buffers must be 16-byte aligned");
    EncodeTiledFn encode = get_encode();
    if (!encode) {
        atvs_set_error("atvs_conv3d_tc: cuTensorMapEncodeTiled entry point not available");
        return ATVS_E_UNSUP;
    }
    cudaStream_t st = (cudaStream_t)stream;
    if (transposed && deconv_ring_supported(Cin, Cout) && deconv_ring_applicable(B, D, H, W)) {
        size_t off = tap_image_bytes(Cin, Cout, 1);
        if (deconv_fused_applicable(Cin, Cout)) off += (deconv_fused_weight_bytes(Cin, Cout) + 255) & ~(size_t)255;
        return deconv_ring(x_bf16, x_dtype, (const char*)wpacked + off, B, D, H, W, Cin, Cout, raw_out, raw16, stats, st);
    }
    if (transposed && deconv_fused_applicable(Cin, Cout))
        return deconv_fused(x_bf16, x_dtype, (const char*)wpacked + tap_image_bytes(Cin, Cout, 1), B, D, H, W, Cin, Cout, raw_out,
                            raw16, stats, st);
    if (!transposed && stride == 2 && ring_s2_applicable(B, D, H, W, Cin, Cout))
        return ring_s2_conv(x_bf16, x_dtype, (const char*)wpacked + tap_image_bytes(Cin, Cout, 0) + ring_weight_bytes(Cin, Cout), B, D, H,
                            W, Cin, Cout, raw_out, raw16, stats, plane_bias, st);
    if (ring_applicable(B, D, H, W, stride, transposed))
        return ring_conv(x_bf16, x_dtype, (const char*)wpacked + tap_image_bytes(Cin, Cout, 0), B, D, H, W, Cin, Cout, raw_out,
                         raw16, stats, plane_bias, st);
    const SlabPlan sp = plan_slabs(Cin, Cout, transposed ? 8 : 27);
    const int ncls = transposed ? 8 : 1;
    const int tps = (Cin == 8) ? 2 : 1;
    const CUtensorMapSwizzle swz = swizzle_for(Cin);
    const char* xb = (const char*)x_bf16;
    size_t wofs = 0;   // element offset into the packed weights

    // transposed convolutions: the 8 output-parity classes share the input, the tile grid and (when the
    // weights of all 27 taps fit one slab) the resident weight image -> ONE launch walks all classes.
    const bool merge = transposed && sp.nslabs == 1;
    const int ngroups = merge ? 1 : ncls;
    for (int grp = 0; grp < ngroups; ++grp) {
        const int c0 = merge ? 0 : grp, c1 = merge ? ncls : grp + 1;
        const ConvGeom g = make_conv_geom(B, D, H, W, Cin, Cout, stride, transposed, c0);
        TcParams p;
        memset(&p, 0, sizeof(p));
        p.B = B; p.Dj = g.Dj; p.Hj = g.Hj; p.Wj = g.Wj;
        p.Do = g.Do; p.Ho = g.Ho; p.Wo = g.Wo;
        p.os = g.os;
        p.Cout = Cout;
        p.raw16 = raw16;
        p.fmt = tc_fmt_bits(x_dtype);
        p.sat = raw16 ? atvs_sat_ptr() : nullptr;
        p.ncls = c1 - c0;
        // brick shape: 128 voxels, minimise padded volume, prefer a wide x extent
        {
            static const int opts[][3] = {{2, 8, 8}, {1, 8, 16}, {4, 4, 8}, {2, 4, 16}, {1, 4, 32}, {4, 8, 4},
                                          {8, 4, 4}, {1, 16, 8}, {2, 16, 4}, {8, 8, 2}, {16, 4, 2}, {32, 2, 2},
                                          {8, 16, 1}, {16, 8, 1}, {128, 1, 1}, {1, 1, 128}, {1, 128, 1}, {1, 2, 64}};
            long long best = -1;
            int bi = 0;
            for (int i = 0; i < (int)(sizeof(opts) / sizeof(opts[0])); ++i) {
                const long long n = (long long)((g.Dj + opts[i][0] - 1) / opts[i][0]) *
                                    ((g.Hj + opts[i][1] - 1) / opts[i][1]) * ((g.Wj + opts[i][2] - 1) / opts[i][2]);
                if (best < 0 || n < best) { best = n; bi = i; }
            }
            const int TD = opts[bi][0], TH = opts[bi][1], TW = opts[bi][2];
            auto lg = [](int v) { int l = 0; while ((1 << l) < v) ++l; return l; };
            p.ltd = lg(TD); p.lth = lg(TH); p.ltw = lg(TW);
            p.nTD = (g.Dj + TD - 1) / TD; p.nTH = (g.Hj + TH - 1) / TH; p.nTW = (g.Wj + TW - 1) / TW;
            p.ntiles = (long long)B * p.nTD * p.nTH * p.nTW;
        }
        const int TD = 1 << p.ltd, TH = 1 << p.lth, TW = 1 << p.ltw;
        // taps of every class in the group, class-major (the packed weights follow the same order)
        int nt = 0;
        for (int cls = c0; cls < c1; ++cls) {
            const ConvGeom gc = make_conv_geom(B, D, H, W, Cin, Cout, stride, transposed, cls);
            p.cls_tap0[cls - c0] = nt;
            for (int a = 0; a < 3; ++a) p.cls_par[cls - c0][a] = gc.p[a];
            for (int tz = 0; tz < gc.nt[0]; ++tz)
                for (int ty = 0; ty < gc.nt[1]; ++ty)
                    for (int tx = 0; tx < gc.nt[2]; ++tx) {
                        const int off[3] = {gc.koff[0][tz], gc.koff[1][ty], gc.koff[2][tx]};
                        TcTap& t = p.taps[nt++];
                        if (gc.s_in == 2) {
                            int par[3], ho[3];
                            for (int a = 0; a < 3; ++a) { par[a] = off[a] & 1; ho[a] = (off[a] - par[a]) / 2; }
                            t.map = (par[0] * 2 + par[1]) * 2 + par[2];
                            t.oz = ho[0]; t.oy = ho[1]; t.ox = ho[2];
                        } else {
                            t.map = 0; t.oz = off[0]; t.oy = off[1]; t.ox = off[2];
                        }
                    }
            while (nt % tps) { p.taps[nt] = p.taps[nt - 1]; ++nt; }   // phantom tap: zero weights
        }
        p.cls_tap0[c1 - c0] = nt;
        p.ntaps = nt;

        // tensor maps over the input
        TcMaps maps;
        memset(&maps, 0, sizeof(maps));
        const int nmaps = (g.s_in == 2) ? 8 : 1;
        for (int m = 0; m < nmaps; ++m) {
            const int pz = (m >> 2) & 1, py = (m >> 1) & 1, px = m & 1;
            const int s = g.s_in;
            cuuint64_t dims[5] = {(cuuint64_t)Cin, (cuuint64_t)(W / s), (cuuint64_t)(H / s), (cuuint64_t)(D / s),
                                  (cuuint64_t)B};
            cuuint64_t strides[4] = {(cuuint64_t)Cin * 2 * s, (cuuint64_t)W * Cin * 2 * s,
                                     (cuuint64_t)H * W * Cin * 2 * s, (cuuint64_t)D * H * W * Cin * 2};
            cuuint32_t box[5] = {(cuuint32_t)Cin, (cuuint32_t)TW, (cuuint32_t)TH, (cuuint32_t)TD, 1};
            cuuint32_t es[5] = {1, 1, 1, 1, 1};
            void* base = (void*)(xb + ((size_t)(pz * H + py) * W + px) * Cin * 2);
            CUresult r = encode(&maps.a[m], CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5, base, dims, strides, box, es,
                                CU_TENSOR_MAP_INTERLEAVE_NONE, swz, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                                CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
            if (r != CUDA_SUCCESS) {
                atvs_set_error("atvs_conv3d_tc: cuTensorMapEncodeTiled(input, map %d) failed: %d", m, (int)r);
                return (int)r;
            }
        }
        for (int slab = 0; slab < sp.nslabs; ++slab) {
            p.coff = slab * sp.npad;
            p.ncols = (Cout - p.coff < sp.npad) ? Cout - p.coff : sp.npad;
            {
                cuuint64_t dims[2] = {(cuuint64_t)Cin, (cuuint64_t)nt * sp.npad};
                cuuint64_t strides[1] = {(cuuint64_t)Cin * 2};
                cuuint32_t box[2] = {(cuuint32_t)Cin, (cuuint32_t)sp.npad};
                cuuint32_t es[2] = {1, 1};
                void* base = (void*)((const char*)wpacked + (wofs + (size_t)slab * nt * sp.npad * Cin) * 2);
                CUresult r = encode(&maps.w, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, base, dims, strides, box, es,
                                    CU_TENSOR_MAP_INTERLEAVE_NONE, swz, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
                if (r != CUDA_SUCCESS) {
                    atvs_set_error("atvs_conv3d_tc: cuTensorMapEncodeTiled(weights) failed: %d", (int)r);
                    return (int)r;
                }
            }
            const size_t wbytes = ((size_t)nt * sp.npad * Cin * 2 + 1023) & ~(size_t)1023;
            const size_t stage_bytes = (size_t)128 * Cin * 2 * tps;
            const size_t budget = 200 * 1024;
            if (wbytes + 2 * stage_bytes > budget) {
                atvs_set_error("atvs_conv3d_tc: weights do not fit in shared memory (Cin=%d Cout=%d)", Cin, Cout);
                return ATVS_E_UNSUP;
            }
            int nst = (int)((budget - wbytes) / stage_bytes);
            if (nst > 8) nst = 8;
            if (nst > nt / tps) nst = nt / tps > 2 ? nt / tps : 2;
            p.nstages = nst;
            const size_t smem = 1024 + wbytes + (size_t)nst * stage_bytes + (2 * nst + 5) * 8 + 16;
            const int sms = atvs_num_sms();
            const long long nwork = p.ntiles * p.ncls;
            const int grid = tc_grid(nwork, sms);
            int rc = 0;
#define TC_CASE(CI, NP) if (Cin == CI && sp.npad == NP) rc = launch_tc<CI, NP>(maps, p, raw_out, stats, plane_bias, smem, grid, st); else
            TC_CASE(8, 16) TC_CASE(16, 16) TC_CASE(16, 32) TC_CASE(32, 16) TC_CASE(32, 32) TC_CASE(32, 64)
            TC_CASE(64, 16) TC_CASE(64, 32) TC_CASE(8, 32) TC_CASE(8, 64) TC_CASE(16, 64) TC_CASE(64, 64)
            {
                atvs_set_error("atvs_conv3d_tc: no kernel for Cin=%d N=%d", Cin, sp.npad);
                return ATVS_E_UNSUP;
            }
#undef TC_CASE
            if (rc) return rc;
        }
        wofs += (size_t)nt * sp.nslabs * sp.npad * Cin;
    }
    return 0;
}


// =========================================================================== 2-D convolutions of the FEM on the same kernel
// tf.layers.conv2d / slim.conv2d (network.py:142-215, 570-599), stride 1, k = 1 | 3, dilation `rate`, TF 'SAME' padding,
// as the D = 1 case of k_conv3d_tc: the input (B,H,W,Cin) is read through one tensor map per chunk of <= 64 input
// channels, a "tap" is (chunk, ky, kx) with the TMA box shifted by ((kx-1)*rate, (ky-1)*rate) (zero fill = padding), and
// all taps' weights of one slab of output channels stay resident in shared memory.  Epilogue: + bias[c], ReLU, raw
// fp32 | saturated fp16 store, optional per-channel moments (conv_bn layers).
namespace {

int conv2d_chunk(int Cin) { return Cin % 64 == 0 ? 64 : (Cin == 32 ? 32 : 0); }

// N tile of a 2-D layer: the largest of {64, 32, 16} covering Cout whose resident weights leave room for >= 3 stages
int conv2d_npad(int Cin, int Cout, int ksize) {
    const int ck = conv2d_chunk(Cin);
    const int ntaps = ksize * ksize * (Cin / ck);
    int npad = Cout <= 16 ? 16 : Cout <= 32 ? 32 : 64;
    while (npad > 16 && (size_t)ntaps * npad * ck * 2 > 150 * 1024) npad >>= 1;
    return npad;
}

// packed image: [slab][tap = (chunk, ky, kx)][NPAD][ck] 16-bit, K-major, from the TF kernel [k,k,Cin,Cout]
__global__ void k_pack_weights2d(const float* __restrict__ w, int Cin, int Cout, int ksize, int ck, int npad, int f16,
                                 unsigned short* __restrict__ out) {
    const int nchunk = Cin / ck, ntaps = ksize * ksize * nchunk;
    const int slab = blockIdx.x / ntaps, tap = blockIdx.x % ntaps;
    const int chunk = tap / (ksize * ksize), kk = tap % (ksize * ksize);
    unsigned short* o = out + ((size_t)slab * ntaps + tap) * npad * ck;
    for (int i = threadIdx.x; i < npad * ck; i += blockDim.x) {
        const int n = i / ck, k = i % ck;
        const int co = slab * npad + n;
        const float val = co < Cout ? w[((size_t)kk * Cin + chunk * ck + k) * Cout + co] : 0.f;
        o[i] = tc_cvt16(val, f16);
    }
}

}  // namespace

extern "C" size_t atvs_packed_weight2d_bytes(int Cin, int Cout, int ksize) {
    const int ck = conv2d_chunk(Cin);
    if (ck == 0 || Cout < 1 || Cout > 256 || !(ksize == 1 || ksize == 3)) return 0;
    const int npad = conv2d_npad(Cin, Cout, ksize);
    const int nslabs = (Cout + npad - 1) / npad;
    return ((size_t)nslabs * ksize * ksize * (Cin / ck) * npad * ck * 2 + 255) & ~(size_t)255;
}

extern "C" int atvs_pack_conv2d_weights_tc(const float* kernel, int Cin, int Cout, int ksize, int dtype, void* wpacked,
                                           atvs_stream_t stream) {
    ATVS_CHECK_ARG(kernel && wpacked, ATVS_E_NULL, "atvs_pack_conv2d_weights_tc: NULL pointer");
    ATVS_CHECK_ARG(dtype == ATVS_BF16 || dtype == ATVS_F16, ATVS_E_DTYPE, "atvs_pack_conv2d_weights_tc: dtype %d", dtype);
    ATVS_CHECK_ARG(atvs_packed_weight2d_bytes(Cin, Cout, ksize) != 0, ATVS_E_UNSUP,
                   "atvs_pack_conv2d_weights_tc: Cin=%d (32 or a multiple of 64) Cout=%d (1..256) k=%d (1 | 3)", Cin, Cout, ksize);
    const int ck = conv2d_chunk(Cin), npad = conv2d_npad(Cin, Cout, ksize);
    const int nslabs = (Cout + npad - 1) / npad, ntaps = ksize * ksize * (Cin / ck);
    k_pack_weights2d<<<nslabs * ntaps, 128, 0, (cudaStream_t)stream>>>(kernel, Cin, Cout, ksize, ck, npad, dtype == ATVS_F16,
                                                                       (unsigned short*)wpacked);
    ATVS_LAUNCH_CHECK();
    return 0;
}

extern "C" int atvs_conv2d_tc(const void* x16, int x_dtype, const void* wpacked, const float* bias, int B, int H, int W,
                              int Cin, int Cout, int ksize, int rate, int relu, void* out, int out_dtype, double* stats,
                              atvs_stream_t stream) {
    ATVS_CHECK_ARG(x16 && wpacked && out, ATVS_E_NULL, "atvs_conv2d_tc: NULL pointer");
    ATVS_CHECK_ARG(x_dtype == ATVS_BF16 || x_dtype == ATVS_F16, ATVS_E_DTYPE, "atvs_conv2d_tc: x_dtype %d", x_dtype);
    ATVS_CHECK_ARG(out_dtype == ATVS_F32 || out_dtype == ATVS_F16, ATVS_E_DTYPE, "atvs_conv2d_tc: out_dtype %d (ATVS_F32 | ATVS_F16)", out_dtype);
    ATVS_CHECK_ARG(B > 0 && H > 0 && W > 0 && rate >= 1, ATVS_E_SHAPE, "atvs_conv2d_tc: bad shape");
    ATVS_CHECK_ARG(atvs_packed_weight2d_bytes(Cin, Cout, ksize) != 0, ATVS_E_UNSUP,
                   "atvs_conv2d_tc: Cin=%d (32 or a multiple of 64) Cout=%d (1..256) k=%d (1 | 3)", Cin, Cout, ksize);
    ATVS_CHECK_ARG((((uintptr_t)x16 | (uintptr_t)wpacked | (uintptr_t)out | (uintptr_t)bias) & 15) == 0, ATVS_E_SHAPE,
                   "atvs_conv2d_tc: buffers must be 16-byte aligned");
    EncodeTiledFn encode = get_encode();
    if (!encode) {
        atvs_set_error("atvs_conv2d_tc: cuTensorMapEncodeTiled entry point not available");
        return ATVS_E_UNSUP;
    }
    cudaStream_t st = (cudaStream_t)stream;
    const int ck = conv2d_chunk(Cin), nchunk = Cin / ck;
    const int npad = conv2d_npad(Cin, Cout, ksize);
    const int nslabs = (Cout + npad - 1) / npad;
    const int nt = ksize * ksize * nchunk;
    ATVS_CHECK_ARG(nt <= TC_MAX_TAPS && nchunk <= 8, ATVS_E_UNSUP, "atvs_conv2d_tc: %d taps (Cin=%d k=%d) exceed %d", nt, Cin,
                   ksize, TC_MAX_TAPS);
    TcParams p;
    memset(&p, 0, sizeof(p));
    p.B = B; p.Dj = 1; p.Hj = H; p.Wj = W;
    p.Do = 1; p.Ho = H; p.Wo = W;
    p.os = 1;
    p.Cout = Cout;
    p.raw16 = out_dtype == ATVS_F16;
    p.fmt = tc_fmt_bits(x_dtype);
    p.sat = p.raw16 ? atvs_sat_ptr() : nullptr;
    p.chan_bias = bias;
    p.relu = relu;
    p.ncls = 1;
    {   // 128-pixel brick: minimise the padded area, prefer wide rows
        static const int opts[][2] = {{8, 16}, {4, 32}, {16, 8}, {2, 64}, {1, 128}, {32, 4}};
        long long best = -1;
        int bi = 0;
        for (int i = 0; i < (int)(sizeof(opts) / sizeof(opts[0])); ++i) {
            const long long n = (long long)((H + opts[i][0] - 1) / opts[i][0]) * ((W + opts[i][1] - 1) / opts[i][1]);
            if (best < 0 || n < best) { best = n; bi = i; }
        }
        auto lg = [](int v) { int l = 0; while ((1 << l) < v) ++l; return l; };
        p.ltd = 0; p.lth = lg(opts[bi][0]); p.ltw = lg(opts[bi][1]);
        p.nTD = 1; p.nTH = (H + opts[bi][0] - 1) / opts[bi][0]; p.nTW = (W + opts[bi][1] - 1) / opts[bi][1];
        p.ntiles = (long long)B * p.nTH * p.nTW;
    }
    const int TH = 1 << p.lth, TW = 1 << p.ltw;
    int n = 0;
    for (int c = 0; c < nchunk; ++c)
        for (int ky = 0; ky < ksize; ++ky)
            for (int kx = 0; kx < ksize; ++kx) {
                TcTap& t = p.taps[n++];
                t.map = c; t.oz = 0;
                t.oy = (ky - ksize / 2) * rate;
                t.ox = (kx - ksize / 2) * rate;
            }
    p.cls_tap0[0] = 0; p.cls_tap0[1] = nt;
    p.ntaps = nt;
    const CUtensorMapSwizzle swz = swizzle_for(ck);
    TcMaps maps;
    memset(&maps, 0, sizeof(maps));
    for (int c = 0; c < nchunk; ++c) {
        cuuint64_t dims[5] = {(cuuint64_t)ck, (cuuint64_t)W, (cuuint64_t)H, 1, (cuuint64_t)B};
        cuuint64_t strides[4] = {(cuuint64_t)Cin * 2, (cuuint64_t)W * Cin * 2, (cuuint64_t)H * W * Cin * 2,
                                 (cuuint64_t)H * W * Cin * 2};
        cuuint32_t box[5] = {(cuuint32_t)ck, (cuuint32_t)TW, (cuuint32_t)TH, 1, 1};
        cuuint32_t es[5] = {1, 1, 1, 1, 1};
        void* base = (void*)((const char*)x16 + (size_t)c * ck * 2);
        CUresult r = encode(&maps.a[c], CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5, base, dims, strides, box, es,
                            CU_TENSOR_MAP_INTERLEAVE_NONE, swz, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) {
            atvs_set_error("atvs_conv2d_tc: cuTensorMapEncodeTiled(input, chunk %d) failed: %d", c, (int)r);
            return (int)r;
        }
    }
    for (int slab = 0; slab < nslabs; ++slab) {
        p.coff = slab * npad;
        p.ncols = (Cout - p.coff < npad) ? Cout - p.coff : npad;
        {
            cuuint64_t dims[2] = {(cuuint64_t)ck, (cuuint64_t)nt * npad};
            cuuint64_t strides[1] = {(cuuint64_t)ck * 2};
            cuuint32_t box[2] = {(cuuint32_t)ck, (cuuint32_t)npad};
            cuuint32_t es[2] = {1, 1};
            void* base = (void*)((const char*)wpacked + (size_t)slab * nt * npad * ck * 2);
            CUresult r = encode(&maps.w, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, base, dims, strides, box, es,
                                CU_TENSOR_MAP_INTERLEAVE_NONE, swz, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                                CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
            if (r != CUDA_SUCCESS) {
                atvs_set_error("atvs_conv2d_tc: cuTensorMapEncodeTiled(weights) failed: %d", (int)r);
                return (int)r;
            }
        }
        const size_t wbytes = ((size_t)nt * npad * ck * 2 + 1023) & ~(size_t)1023;
        const size_t stage_bytes = (size_t)128 * ck * 2;
        const size_t budget = 216 * 1024;
        if (wbytes + 2 * stage_bytes > budget) {
            atvs_set_error("atvs_conv2d_tc: weights do not fit in shared memory (Cin=%d Cout=%d k=%d)", Cin, Cout, ksize);
            return ATVS_E_UNSUP;
        }
        int nst = (int)((budget - wbytes) / stage_bytes);
        if (nst > 8) nst = 8;
        if (nst > nt) nst = nt > 2 ? nt : 2;
        p.nstages = nst;
        const size_t smem = 1024 + wbytes + (size_t)nst * stage_bytes + (2 * nst + 5) * 8 + 16;
        const int sms = atvs_num_sms();
        const int grid = (int)(p.ntiles < sms ? p.ntiles : sms);
        int rc = 0;
        if (ck == 32 && npad == 16) rc = launch_tc<32, 16>(maps, p, (float*)out, stats, nullptr, smem, grid, st);
        else if (ck == 32 && npad == 32) rc = launch_tc<32, 32>(maps, p, (float*)out, stats, nullptr, smem, grid, st);
        else if (ck == 32 && npad == 64) rc = launch_tc<32, 64>(maps, p, (float*)out, stats, nullptr, smem, grid, st);
        else if (ck == 64 && npad == 16) rc = launch_tc<64, 16>(maps, p, (float*)out, stats, nullptr, smem, grid, st);
        else if (ck == 64 && npad == 32) rc = launch_tc<64, 32>(maps, p, (float*)out, stats, nullptr, smem, grid, st);
        else rc = launch_tc<64, 64>(maps, p, (float*)out, stats, nullptr, smem, grid, st);
        if (rc) return rc;
    }
    return 0;
}
