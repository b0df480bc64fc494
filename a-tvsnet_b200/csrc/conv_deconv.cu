// conv_deconv.cu - stride-2 transposed 3x3x3 convolution (network.py:511-550 deconv_bn,
// tf.layers.conv3d_transpose 'SAME': out[2i+k] += in[i]*w[k]) as a tcgen05 implicit GEMM in which
// ALL 8 output-parity classes of an input tile are produced together.
//
//   tile        = 128 input voxels j (brick TD x TH x TW); its outputs are the 8 x 128 voxels 2j + p
//   A tiles     = the 8 shifted input bricks (offsets in {0,-1}^3), one TMA box load each (zero fill
//                 outside the volume), instead of one load per (class, tap) pair (27);
//   MMAs        = the 27 (class, tap) products, grouped by the shift they read: shift s feeds every
//                 class whose tap list contains that offset, each into its own TMEM accumulator
//                 (8 classes x N columns, double buffered) with that pair's weight tile;
//   epilogue    = per class: tcgen05.ld -> raw fp32 store at the parity position + BN moments.
//   One pipeline round trip (barriers, commits, epilogue wake-up) per 1024 outputs instead of per
//   128: the per-class formulation was bound by that fixed cost, not by the tensor pipe.
#include "tc_ptx.cuh"
#include "conv_deconv.cuh"
#include <cstring>

namespace {

constexpr int DC_THREADS = 192;

struct DcParams {
    int B, Dj, Hj, Wj;             // input extent (= iteration space)
    int ltd, lth, ltw, nTD, nTH, nTW;
    int Cout, ncols;
    int raw16;                     // raw output dtype: 0 fp32, 1 saturated fp16
    uint32_t fmt;                  // operand format bits of the instruction descriptor (tc_fmt_bits)
    unsigned long long* sat;       // saturation counter of the fp16 raw stores (atvs_sat_ptr)
    int nstages;
    int sh_off[8][3];              // shift s reads input voxel j + sh_off[s]
    int sh_first[9];               // pairs of shift s are [sh_first[s], sh_first[s+1])
    int pair_cls[27];              // output parity class (pz*4 + py*2 + px) of each pair
    int pair_init[27];             // 1 = first product into that class' accumulator (overwrite)
    long long ntiles;
};

struct alignas(64) DcMaps {
    CUtensorMap a;
    CUtensorMap w;
};

template <int CIN>
struct DcCfg {
    static constexpr int KSTEPS = CIN / 16;
    static constexpr int TILE_BYTES = 128 * CIN * 2;
    static constexpr uint32_t LAYOUT = (CIN == 64) ? 2u : (CIN == 32) ? 4u : 6u;
    static constexpr uint32_t SBO = (uint32_t)(8 * CIN * 2);
};

// Cin = 16, N = 16: 256 TMEM columns and < 100 KB of shared memory per CTA -> two CTAs per SM, which
// doubles the epilogue throughput (the 8-class epilogue, not the tensor pipe, bounds this instance)
template <int CIN, int NPAD>
struct DcOcc {
    static constexpr int MINB = (CIN == 16 && NPAD == 16) ? 2 : 1;
};

template <int CIN, int NPAD>
__global__ void __launch_bounds__(DC_THREADS, DcOcc<CIN, NPAD>::MINB)
k_deconv3d_tc(const __grid_constant__ DcMaps tm, const __grid_constant__ DcParams p, float* __restrict__ out,
              double* __restrict__ stats) {
    using Cfg = DcCfg<CIN>;
    constexpr int WPAIR_BYTES = NPAD * CIN * 2;
    constexpr uint32_t ACC_COLS = 8 * NPAD;                 // one accumulator set (8 classes)
    constexpr uint32_t TMEM_COLS = 2 * ACC_COLS;            // double buffered: 256 (N=16) or 512 (N=32)
    const uint32_t IDESC = (1u << 4) | ((uint32_t)(NPAD >> 3) << 17) | ((128u >> 4) << 24) | p.fmt;

    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    uint8_t* wsm = smem;
    const int wbytes = 27 * WPAIR_BYTES;
    uint8_t* asmem = smem + ((wbytes + 1023) & ~1023);
    uint64_t* bars = reinterpret_cast<uint64_t*>(asmem + (size_t)p.nstages * Cfg::TILE_BYTES);
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

    if (warp == 0) {
        // ===================== TMA producer (converged warp, elected lane issues) =====================
        const uint32_t leader = elect_one();
        mbar_expect_tx_leader(wbar, (uint32_t)wbytes, leader);
        for (int t = 0; t < 27; ++t) tma_load_2d_leader(wsm + (size_t)t * WPAIR_BYTES, &tm.w, 0, t * NPAD, wbar, leader);
        int stage = 0;
        uint32_t phase = 0;
        for (long long tile = blockIdx.x; tile < p.ntiles; tile += gridDim.x) {
            const int b = (int)(tile / tiles_per_b);
            int r = (int)(tile % tiles_per_b);
            const int jx0 = (r % p.nTW) << p.ltw;
            r /= p.nTW;
            const int jy0 = (r % p.nTH) << p.lth;
            const int jz0 = (r / p.nTH) << p.ltd;
            for (int s = 0; s < 8; ++s) {
                mbar_wait(&empty[stage], phase ^ 1);
                mbar_expect_tx_leader(&full[stage], (uint32_t)Cfg::TILE_BYTES, leader);
                tma_load_5d_leader(asmem + (size_t)stage * Cfg::TILE_BYTES, &tm.a, 0, jx0 + p.sh_off[s][2],
                                   jy0 + p.sh_off[s][1], jz0 + p.sh_off[s][0], b, &full[stage], leader);
                if (++stage == p.nstages) {
                    stage = 0;
                    phase ^= 1;
                }
            }
        }
    } else if (warp == 1) {
        // ===================== MMA issuer (converged warp, elected lane issues) =====================
        const uint32_t leader = elect_one();
        mbar_wait(wbar, 0);
        tc_fence_after();
        const uint64_t wdesc0 = make_desc(smem_u32(wsm), 16u, Cfg::SBO, Cfg::LAYOUT);
        int stage = 0;
        uint32_t phase = 0;
        long long it = 0;
        for (long long tile = blockIdx.x; tile < p.ntiles; tile += gridDim.x, ++it) {
            const int acc = (int)(it & 1);
            mbar_wait(&tempty[acc], (uint32_t)(((it >> 1) & 1) ^ 1));
            tc_fence_after();
            const uint32_t dbase = tmem_base + (uint32_t)acc * ACC_COLS;
            for (int s = 0; s < 8; ++s) {
                mbar_wait(&full[stage], phase);
                tc_fence_after();
                const uint64_t ad0 = make_desc(smem_u32(asmem + (size_t)stage * Cfg::TILE_BYTES), 16u, Cfg::SBO, Cfg::LAYOUT);
                for (int pr = p.sh_first[s]; pr < p.sh_first[s + 1]; ++pr) {
                    const uint32_t dcol = dbase + (uint32_t)(p.pair_cls[pr] * NPAD);
                    const uint64_t bd0 = desc_advance(wdesc0, (uint32_t)(pr * WPAIR_BYTES));
                    const bool init = p.pair_init[pr] != 0;
#pragma unroll
                    for (int ks = 0; ks < Cfg::KSTEPS; ++ks) {
                        const uint64_t ad = desc_advance(ad0, ks * 32), bd = desc_advance(bd0, ks * 32);
                        if (ks == 0 && init) tc_mma_bf16_first(dcol, ad, bd, IDESC, leader);
                        else tc_mma_bf16_acc(dcol, ad, bd, IDESC, leader);
                    }
                }
                tc_commit_leader(&empty[stage], leader);
                if (++stage == p.nstages) {
                    stage = 0;
                    phase ^= 1;
                }
            }
            tc_commit_leader(&tfull[acc], leader);
        }
    } else {
        // ===================== epilogue (4 warps = 128 TMEM lanes), 8 classes per tile =====================
        const int g = warp & 3;
        const int row = g * 32 + lane;
        const int tw = row & ((1 << p.ltw) - 1);
        const int th = (row >> p.ltw) & ((1 << p.lth) - 1);
        const int td = row >> (p.ltw + p.lth);
        float run[2 * NPAD];
#pragma unroll
        for (int i = 0; i < 2 * NPAD; ++i) run[i] = 0.f;
        const int vec = raw_vec_mode(out, p.ncols, p.Cout, 0);
        const int Do = 2 * p.Dj, Ho = 2 * p.Hj, Wo = 2 * p.Wj;
        long long it = 0;
        for (long long tile = blockIdx.x; tile < p.ntiles; tile += gridDim.x, ++it) {
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
            const uint32_t taddr = tmem_base + ((uint32_t)(g * 32) << 16) + (uint32_t)acc * ACC_COLS;
#pragma unroll 1
            for (int cls = 0; cls < 8; ++cls) {
                const int pz = cls >> 2, py = (cls >> 1) & 1, px = cls & 1;
                const size_t o = valid ? ((((size_t)b * Do + (2 * jz + pz)) * Ho + (2 * jy + py)) * Wo + (2 * jx + px)) * p.Cout : 0;
                // the accumulator set is released after the LAST class has been read
                epilogue_tile<NPAD>(taddr + (uint32_t)(cls * NPAD), cls == 7 ? &tempty[acc] : nullptr, lane, valid, out, o,
                                    p.ncols, vec, p.raw16, stats != nullptr, run, nullptr, p.sat);
            }
        }
        if (stats != nullptr) flush_stats<NPAD>(stats, run, lane, p.Cout, 0, p.ncols);
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
    }
}

// shift-major list of the 27 (class, tap) pairs
struct PairTable {
    int sh_off[8][3];
    int sh_first[9];
    int pair_cls[27];
    int pair_kidx[27];
    int pair_init[27];
};

__host__ __device__ inline PairTable make_pair_table() {
    PairTable t;
    bool seen[8] = {false, false, false, false, false, false, false, false};
    int n = 0;
    for (int s = 0; s < 8; ++s) {
        const int off[3] = {-((s >> 2) & 1), -((s >> 1) & 1), -(s & 1)};
        for (int a = 0; a < 3; ++a) t.sh_off[s][a] = off[a];
        t.sh_first[s] = n;
        for (int cls = 0; cls < 8; ++cls) {
            const int par[3] = {(cls >> 2) & 1, (cls >> 1) & 1, cls & 1};
            int k[3];
            bool ok = true;
            for (int a = 0; a < 3; ++a) {
                // parity 0: taps (k=0, off 0), (k=2, off -1); parity 1: tap (k=1, off 0)
                if (par[a] == 0) k[a] = (off[a] == 0) ? 0 : 2;
                else if (off[a] == 0) k[a] = 1;
                else ok = false;
            }
            if (!ok) continue;
            t.pair_cls[n] = cls;
            t.pair_kidx[n] = (k[0] * 3 + k[1]) * 3 + k[2];
            t.pair_init[n] = seen[cls] ? 0 : 1;
            seen[cls] = true;
            ++n;
        }
    }
    t.sh_first[8] = n;   // == 27
    return t;
}

// weight image: [27 pairs, shift-major][NPAD rows (co)][Cin (k)] bf16 from the TF kernel [3,3,3,Cout,Cin]
__global__ void k_pack_deconv(const float* __restrict__ w, int Cin, int Cout, int npad, int f16, unsigned short* __restrict__ out) {
    const PairTable t = make_pair_table();
    const int pr = blockIdx.x;
    const int kidx = t.pair_kidx[pr];
    unsigned short* o = out + (size_t)pr * npad * Cin;
    for (int i = threadIdx.x; i < npad * Cin; i += blockDim.x) {
        const int n = i / Cin, k = i % Cin;
        o[i] = tc_cvt16(n < Cout ? w[((size_t)kidx * Cout + n) * Cin + k] : 0.f, f16);
    }
}

template <int CIN, int NPAD>
int launch_dc(const DcMaps& maps, const DcParams& p, float* out, double* stats, size_t smem, int grid, cudaStream_t st) {
    if (const int rc = atvs_max_dynamic_smem<k_deconv3d_tc<CIN, NPAD>>()) return rc;
    k_deconv3d_tc<CIN, NPAD><<<grid, DC_THREADS, smem, st>>>(maps, p, out, stats);
    ATVS_LAUNCH_CHECK();
    return 0;
}

}  // namespace

static int deconv_npad(int Cout) { return Cout <= 16 ? 16 : 32; }

bool deconv_fused_applicable(int Cin, int Cout) {
    if (!(Cin == 16 || Cin == 32 || Cin == 64) || Cout > 32) return false;
    const size_t wbytes = ((size_t)27 * deconv_npad(Cout) * Cin * 2 + 1023) & ~(size_t)1023;
    return wbytes + 3 * (size_t)128 * Cin * 2 <= 200 * 1024;
}

size_t deconv_fused_weight_bytes(int Cin, int Cout) { return (size_t)27 * deconv_npad(Cout) * Cin * 2; }

int deconv_fused_pack(const float* kernel, int Cin, int Cout, int dtype, void* wimg, cudaStream_t st) {
    k_pack_deconv<<<27, 128, 0, st>>>(kernel, Cin, Cout, deconv_npad(Cout), dtype == ATVS_F16, (unsigned short*)wimg);
    ATVS_LAUNCH_CHECK();
    return 0;
}

int deconv_fused(const void* x_bf16, int dtype, const void* wimg, int B, int D, int H, int W, int Cin, int Cout, float* raw_out,
                 int raw16, double* stats, cudaStream_t st) {
    EncodeTiledFn encode = get_encode();
    if (!encode) {
        atvs_set_error("atvs_conv3d_bf16: cuTensorMapEncodeTiled entry point not available");
        return ATVS_E_UNSUP;
    }
    const int npad = deconv_npad(Cout);
    DcParams p;
    memset(&p, 0, sizeof(p));
    p.B = B; p.Dj = D; p.Hj = H; p.Wj = W; p.Cout = Cout; p.ncols = Cout;
    p.raw16 = raw16;
    p.fmt = tc_fmt_bits(dtype);
    p.sat = raw16 ? atvs_sat_ptr() : nullptr;
    {
        static const int opts[][3] = {{2, 8, 8}, {1, 8, 16}, {4, 4, 8}, {2, 4, 16}, {1, 4, 32}, {4, 8, 4}, {8, 4, 4},
                                      {1, 16, 8}, {2, 16, 4}, {8, 8, 2}, {16, 4, 2}, {32, 2, 2}, {8, 16, 1}, {16, 8, 1},
                                      {128, 1, 1}, {1, 1, 128}, {1, 128, 1}, {1, 2, 64}};
        long long best = -1;
        int bi = 0;
        for (int i = 0; i < (int)(sizeof(opts) / sizeof(opts[0])); ++i) {
            const long long n = (long long)((D + opts[i][0] - 1) / opts[i][0]) * ((H + opts[i][1] - 1) / opts[i][1]) *
                                ((W + opts[i][2] - 1) / opts[i][2]);
            if (best < 0 || n < best) { best = n; bi = i; }
        }
        const int TD = opts[bi][0], TH = opts[bi][1], TW = opts[bi][2];
        auto lg = [](int v) { int l = 0; while ((1 << l) < v) ++l; return l; };
        p.ltd = lg(TD); p.lth = lg(TH); p.ltw = lg(TW);
        p.nTD = (D + TD - 1) / TD; p.nTH = (H + TH - 1) / TH; p.nTW = (W + TW - 1) / TW;
        p.ntiles = (long long)B * p.nTD * p.nTH * p.nTW;
    }
    const PairTable t = make_pair_table();
    memcpy(p.sh_off, t.sh_off, sizeof(p.sh_off));
    memcpy(p.sh_first, t.sh_first, sizeof(p.sh_first));
    memcpy(p.pair_cls, t.pair_cls, sizeof(p.pair_cls));
    memcpy(p.pair_init, t.pair_init, sizeof(p.pair_init));

    const CUtensorMapSwizzle swz = Cin == 64 ? CU_TENSOR_MAP_SWIZZLE_128B
                                 : Cin == 32 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B;
    DcMaps maps;
    memset(&maps, 0, sizeof(maps));
    {
        cuuint64_t dims[5] = {(cuuint64_t)Cin, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)D, (cuuint64_t)B};
        cuuint64_t strides[4] = {(cuuint64_t)Cin * 2, (cuuint64_t)W * Cin * 2, (cuuint64_t)H * W * Cin * 2,
                                 (cuuint64_t)D * H * W * Cin * 2};
        cuuint32_t box[5] = {(cuuint32_t)Cin, 1u << p.ltw, 1u << p.lth, 1u << p.ltd, 1};
        cuuint32_t es[5] = {1, 1, 1, 1, 1};
        CUresult r = encode(&maps.a, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5, const_cast<void*>(x_bf16), dims, strides, box, es,
                            CU_TENSOR_MAP_INTERLEAVE_NONE, swz, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) {
            atvs_set_error("atvs_conv3d_bf16(deconv): cuTensorMapEncodeTiled(input) failed: %d", (int)r);
            return (int)r;
        }
    }
    {
        cuuint64_t dims[2] = {(cuuint64_t)Cin, (cuuint64_t)27 * npad};
        cuuint64_t strides[1] = {(cuuint64_t)Cin * 2};
        cuuint32_t box[2] = {(cuuint32_t)Cin, (cuuint32_t)npad};
        cuuint32_t es[2] = {1, 1};
        CUresult r = encode(&maps.w, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(wimg), dims, strides, box, es,
                            CU_TENSOR_MAP_INTERLEAVE_NONE, swz, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) {
            atvs_set_error("atvs_conv3d_bf16(deconv): cuTensorMapEncodeTiled(weights) failed: %d", (int)r);
            return (int)r;
        }
    }
    const size_t wbytes = ((size_t)27 * npad * Cin * 2 + 1023) & ~(size_t)1023;
    const size_t stage_bytes = (size_t)128 * Cin * 2;
    const int minb = (Cin == 16 && npad == 16) ? 2 : 1;
    int nst = (int)(((minb == 2 ? 100 : 200) * 1024 - wbytes) / stage_bytes);
    if (nst > 16) nst = 16;
    p.nstages = nst;
    const size_t smem = 1024 + wbytes + (size_t)nst * stage_bytes + (2 * nst + 5) * 8 + 16;
    const int sms = atvs_num_sms();
    const int grid = (int)(p.ntiles < (long long)sms * minb ? p.ntiles : (long long)sms * minb);
#define DC_CASE(CI, NP) if (Cin == CI && npad == NP) return launch_dc<CI, NP>(maps, p, raw_out, stats, smem, grid, st);
    DC_CASE(16, 16) DC_CASE(16, 32) DC_CASE(32, 16) DC_CASE(32, 32) DC_CASE(64, 16) DC_CASE(64, 32)
#undef DC_CASE
    atvs_set_error("atvs_conv3d_bf16(deconv): no kernel for Cin=%d N=%d", Cin, npad);
    return ATVS_E_UNSUP;
}
