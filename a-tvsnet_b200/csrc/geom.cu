// geom.cu - plane-sweep geometry kernels of libatvs.so (compiled with --fmad=false).
//
//   atvs_get_homographies            <- homography_warping.py:179-227
//   atvs_homography_warping          <- homography_warping.py:230-271 + interpolate :31-104
//   atvs_homography_warping_by_depth <- homography_warping.py:108-176
//   atvs_build_cost_volume           <- model.py:157-200 (and the L1 variant :272-280)
//   atvs_prob2depth                  <- model.py:80-129, 13-76
//
// The coordinate arithmetic uses explicit round-to-nearest intrinsics in the order the CPU
// oracle documents (oracle/homography_warping.py), so homographies, sample coordinates,
// floor() cells and validity masks are bit-identical to the oracle; only the last blend may
// differ by rounding of the products (it does not: same order, no FMA).
#include "common.cuh"
#include <cstdlib>
#include <type_traits>

#define MUL(a, b) __fmul_rn((a), (b))
#define ADD(a, b) __fadd_rn((a), (b))
#define SUB(a, b) __fsub_rn((a), (b))
#define DIV(a, b) __fdiv_rn((a), (b))

namespace {

__device__ __forceinline__ float dot3(float a0, float b0, float a1, float b1, float a2, float b2) {
    return ADD(ADD(MUL(a0, b0), MUL(a1, b1)), MUL(a2, b2));
}

struct M3 {
    float m[3][3];
};

__device__ __forceinline__ M3 mm3(const M3& a, const M3& b) {
    M3 r;
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j)
            r.m[i][j] = dot3(a.m[i][0], b.m[0][j], a.m[i][1], b.m[1][j], a.m[i][2], b.m[2][j]);
    return r;
}

__device__ __forceinline__ M3 inv3(const M3& k) {
    const float a = k.m[0][0], b = k.m[0][1], c = k.m[0][2];
    const float d = k.m[1][0], e = k.m[1][1], f = k.m[1][2];
    const float g = k.m[2][0], h = k.m[2][1], i = k.m[2][2];
    const float c00 = SUB(MUL(e, i), MUL(f, h));
    const float c01 = SUB(MUL(d, i), MUL(f, g));
    const float c02 = SUB(MUL(d, h), MUL(e, g));
    const float det = ADD(SUB(MUL(a, c00), MUL(b, c01)), MUL(c, c02));
    M3 r;
    r.m[0][0] = DIV(c00, det);
    r.m[0][1] = DIV(SUB(MUL(c, h), MUL(b, i)), det);
    r.m[0][2] = DIV(SUB(MUL(b, f), MUL(c, e)), det);
    r.m[1][0] = DIV(SUB(MUL(f, g), MUL(d, i)), det);
    r.m[1][1] = DIV(SUB(MUL(a, i), MUL(c, g)), det);
    r.m[1][2] = DIV(SUB(MUL(c, d), MUL(a, f)), det);
    r.m[2][0] = DIV(c02, det);
    r.m[2][1] = DIV(SUB(MUL(b, g), MUL(a, h)), det);
    r.m[2][2] = DIV(SUB(MUL(a, e), MUL(b, d)), det);
    return r;
}

struct Cam {
    M3 R, K;
    float t[3];
};

__device__ __forceinline__ Cam load_cam(const float* cam) {  // (2,4,4) row-major
    Cam c;
#pragma unroll
    for (int i = 0; i < 3; ++i) {
#pragma unroll
        for (int j = 0; j < 3; ++j) {
            c.R.m[i][j] = cam[i * 4 + j];
            c.K.m[i][j] = cam[16 + i * 4 + j];
        }
        c.t[i] = cam[i * 4 + 3];
    }
    return c;
}

__device__ __forceinline__ M3 transpose3(const M3& a) {
    M3 r;
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j) r.m[i][j] = a.m[j][i];
    return r;
}

// c = -(R^T t)
__device__ __forceinline__ void centre(const M3& Rt, const float* t, float* c) {
#pragma unroll
    for (int i = 0; i < 3; ++i) c[i] = -dot3(Rt.m[i][0], t[0], Rt.m[i][1], t[1], Rt.m[i][2], t[2]);
}

__global__ void k_get_homographies(const float* __restrict__ lcam, const float* __restrict__ rcam, int B, int D,
                                   const float* __restrict__ dstart, const float* __restrict__ dint,
                                   int inverse_depth, float* __restrict__ out) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= B * D) return;
    const int b = idx / D, d = idx % D;
    const Cam L = load_cam(lcam + (size_t)b * 32), R = load_cam(rcam + (size_t)b * 32);
    const float depth = ADD(dstart[b], MUL((float)d, dint[b]));
    const M3 Kli = inv3(L.K);
    const M3 RlT = transpose3(L.R), RrT = transpose3(R.R);
    float cl[3], cr[3];
    centre(RlT, L.t, cl);
    centre(RrT, R.t, cr);
    M3 m0;
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        const float crel = SUB(cr[i], cl[i]);
#pragma unroll
        for (int j = 0; j < 3; ++j) {
            const float tv = MUL(crel, L.R.m[2][j]);
            const float sc = inverse_depth ? MUL(tv, depth) : DIV(tv, depth);
            m0.m[i][j] = SUB(i == j ? 1.0f : 0.0f, sc);
        }
    }
    const M3 m1 = mm3(RlT, Kli);
    const M3 m2 = mm3(m0, m1);
    const M3 Hm = mm3(R.K, mm3(R.R, m2));
    float* o = out + (size_t)idx * 9;
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j) o[i * 3 + j] = Hm.m[i][j];
}

// ------------------------------------------------------------------ sampling helpers
struct Sample {
    int x0, y0;            // top-left cell (valid only)
    float wa, wb, wc, wd;  // bilinear areas
    bool valid;
    bool finite;
};

// (u, v) texture coordinates -> bilinear cell, homography_warping.py:37-43,59-95
__device__ __forceinline__ Sample make_sample(float u, float v, int H, int W) {
    Sample s;
    const float x = SUB(u, 0.5f), y = SUB(v, 0.5f);
    s.valid = (x >= 0.0f) && (y >= 0.0f) && (x < (float)(W - 1)) && (y < (float)(H - 1)) && !isnan(x) && !isnan(y);
    s.finite = isfinite(x) && isfinite(y);
    if (s.valid) {
        const float fx = floorf(x), fy = floorf(y);
        s.x0 = (int)fx;
        s.y0 = (int)fy;
        const float x1 = (float)(s.x0 + 1), y1 = (float)(s.y0 + 1);
        const float dx1 = SUB(x1, x), dx0 = SUB(x, fx), dy1 = SUB(y1, y), dy0 = SUB(y, fy);
        s.wa = MUL(dy1, dx1);
        s.wb = MUL(dy1, dx0);
        s.wc = MUL(dy0, dx1);
        s.wd = MUL(dy0, dx0);
    } else {
        s.x0 = s.y0 = 0;
        s.wa = s.wb = s.wc = s.wd = 0.0f;
    }
    return s;
}

__device__ __forceinline__ void homography_uv(const float* __restrict__ h, int x, int y, float& u, float& v) {
    const float px = ADD((float)x, 0.5f), py = ADD((float)y, 0.5f);
    const float xa = ADD(ADD(MUL(h[0], px), MUL(h[1], py)), h[2]);
    const float ya = ADD(ADD(MUL(h[3], px), MUL(h[4], py)), h[5]);
    float z = ADD(ADD(MUL(h[6], px), MUL(h[7], py)), h[8]);
    z = ADD(z, (z == 0.0f) ? 1e-7f : 0.0f);
    u = DIV(xa, z);
    v = DIV(ya, z);
}

__device__ __forceinline__ float blend(const Sample& s, float a, float b, float c, float d) {
    return ADD(ADD(ADD(MUL(s.wa, a), MUL(s.wb, b)), MUL(s.wc, c)), MUL(s.wd, d));
}

__device__ __forceinline__ float4 sample4(const Sample& s, const float* __restrict__ img, int W, int C, int c0) {
    // img points at the (H,W,C) image of this batch element
    if (!s.valid) {
        const float z = s.finite ? 0.0f : __int_as_float(0x7fc00000);
        return make_float4(z, z, z, z);
    }
    const float* p = img + ((size_t)s.y0 * W + s.x0) * C + c0;
    const float4 a = __ldg(reinterpret_cast<const float4*>(p));
    const float4 b = __ldg(reinterpret_cast<const float4*>(p + C));
    const float4 c = __ldg(reinterpret_cast<const float4*>(p + (size_t)W * C));
    const float4 d = __ldg(reinterpret_cast<const float4*>(p + (size_t)W * C + C));
    return make_float4(blend(s, a.x, b.x, c.x, d.x), blend(s, a.y, b.y, c.y, d.y), blend(s, a.z, b.z, c.z, d.z),
                       blend(s, a.w, b.w, c.w, d.w));
}

__device__ __forceinline__ float sample1(const Sample& s, const float* __restrict__ img, int W, int C, int c) {
    if (!s.valid) return s.finite ? 0.0f : __int_as_float(0x7fc00000);
    const float* p = img + ((size_t)s.y0 * W + s.x0) * C + c;
    return blend(s, __ldg(p), __ldg(p + C), __ldg(p + (size_t)W * C), __ldg(p + (size_t)W * C + C));
}

// nearest: homography_warping.py:45-56 (no zeroing: invalid pixels read image[0,0])
__device__ __forceinline__ void nearest_cell(float u, float v, int H, int W, int& x0, int& y0, bool& valid) {
    const float x = SUB(u, 0.5f), y = SUB(v, 0.5f);
    valid = (x >= 0.0f) && (y >= 0.0f) && (x < (float)(W - 1)) && (y < (float)(H - 1)) && !isnan(x) && !isnan(y);
    x0 = valid ? __float2int_rn(x) : 0;   // round half to even == tf.round
    y0 = valid ? __float2int_rn(y) : 0;
}

// ------------------------------------------------------------------ warping kernels
// one thread = one pixel x VEC channels.  BYDEPTH: per-pixel inverse depth instead of H.
template <int VEC, bool BYDEPTH>
__global__ void k_warp(const float* __restrict__ img, const float* __restrict__ hmat, const float* __restrict__ depth,
                       int inverse_depth, int B, int H, int W, int C, int method, float* __restrict__ out,
                       uint8_t* __restrict__ mask) {
    const int G = C / VEC;
    const long long total = (long long)B * H * W * G;
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= total) return;
    const int g = (int)(idx % G);
    const long long pix = idx / G;
    const int x = (int)(pix % W);
    const int y = (int)((pix / W) % H);
    const int b = (int)(pix / ((long long)W * H));
    float u, v;
    if (BYDEPTH) {
        // hmat = (B,12): mat (9) then vec (3), prepared by k_bydepth_setup
        const float* m = hmat + (size_t)b * 12;
        const float dep = depth[pix];
        const float px = ADD((float)x, 0.5f), py = ADD((float)y, 0.5f);
        float q[3];
#pragma unroll
        for (int r = 0; r < 3; ++r) {
            const float vv = inverse_depth ? MUL(m[9 + r], dep) : DIV(m[9 + r], dep);
            q[r] = ADD(ADD(ADD(MUL(m[r * 3], px), MUL(m[r * 3 + 1], py)), m[r * 3 + 2]), vv);
        }
        u = DIV(q[0], q[2]);
        v = DIV(q[1], q[2]);
    } else {
        homography_uv(hmat + (size_t)b * 9, x, y, u, v);
    }
    const float* im = img + (size_t)b * H * W * C;
    if (method == 1) {
        int x0, y0;
        bool valid;
        nearest_cell(u, v, H, W, x0, y0, valid);
        const float* p = im + ((size_t)y0 * W + x0) * C + g * VEC;
        float* o = out + pix * C + g * VEC;
#pragma unroll
        for (int i = 0; i < VEC; ++i) o[i] = __ldg(p + i);
        if (mask && g == 0) mask[pix] = valid ? 1 : 0;
        return;
    }
    const Sample s = make_sample(u, v, H, W);
    if (VEC == 4) {
        *reinterpret_cast<float4*>(out + pix * C + g * 4) = sample4(s, im, W, C, g * 4);
    } else {
        out[pix * C + g] = sample1(s, im, W, C, g);
    }
    if (mask && g == 0) mask[pix] = s.valid ? 1 : 0;
}

// homography_warping.py:115-146: mat = Kr (Rr (Rl^T Kl^-1)), vec = Kr (Rr c_l) + Kr t_r
__global__ void k_bydepth_setup(const float* __restrict__ lcam, const float* __restrict__ rcam, int B,
                                float* __restrict__ mv) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    const Cam L = load_cam(lcam + (size_t)b * 32), R = load_cam(rcam + (size_t)b * 32);
    const M3 RlT = transpose3(L.R);
    float cl[3];
    centre(RlT, L.t, cl);
    const M3 mat = mm3(R.K, mm3(R.R, mm3(RlT, inv3(L.K))));
    float rc[3], v1[3], v2[3];
#pragma unroll
    for (int i = 0; i < 3; ++i) rc[i] = dot3(R.R.m[i][0], cl[0], R.R.m[i][1], cl[1], R.R.m[i][2], cl[2]);
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        v1[i] = dot3(R.K.m[i][0], rc[0], R.K.m[i][1], rc[1], R.K.m[i][2], rc[2]);
        v2[i] = dot3(R.K.m[i][0], R.t[0], R.K.m[i][1], R.t[1], R.K.m[i][2], R.t[2]);
    }
    float* o = mv + (size_t)b * 12;
#pragma unroll
    for (int i = 0; i < 3; ++i) {
#pragma unroll
        for (int j = 0; j < 3; ++j) o[i * 3 + j] = mat.m[i][j];
        o[9 + i] = ADD(v1[i], v2[i]);
    }
}

// ------------------------------------------------------------------ fused cost volume (K1)
__device__ __forceinline__ void store4(float* p, float4 v) { __stcs(reinterpret_cast<float4*>(p), v); }
__device__ __forceinline__ void store4(__nv_bfloat16* p, float4 v) {
    __nv_bfloat162 lo = __floats2bfloat162_rn(v.x, v.y), hi = __floats2bfloat162_rn(v.z, v.w);
    uint2 pk;
    pk.x = *reinterpret_cast<unsigned*>(&lo);
    pk.y = *reinterpret_cast<unsigned*>(&hi);
    __stcs(reinterpret_cast<uint2*>(p), pk);
}
__device__ __forceinline__ unsigned f16x2_sat(float lo, float hi) {
    unsigned r;
    asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
    return r;
}
__device__ __forceinline__ void store4(__half* p, float4 v) {
    uint2 pk;
    pk.x = f16x2_sat(v.x, v.y);
    pk.y = f16x2_sat(v.z, v.w);
    __stcs(reinterpret_cast<uint2*>(p), pk);
}

constexpr int K1_DCHUNK = 8;      // depth planes per block of K1 (measured: 4 / 8 / 16, see DESIGN.md)

// grid: x = pixel*channel-group tiles, y = depth chunks, z = batch.
// one thread = one pixel x 4 channels, looping over K1_DCHUNK planes with the reference
// float4 kept in registers; every plane's slice goes straight to HBM with streaming stores.
template <typename OutT, int MODE, bool WARP_REF>
__global__ void __launch_bounds__(256)
k_build_cost_volume_generic(const float* __restrict__ ref, const float* __restrict__ view, const float* __restrict__ hv,
                    const float* __restrict__ hr, int D, int h, int w, int F, OutT* __restrict__ out) {
    const int G = F >> 2;
    const int hw = h * w;
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= hw * G) return;
    const int g = idx % G, pix = idx / G;
    const int x = pix % w, y = pix / w;
    const int b = blockIdx.z;
    const float* refb = ref + (size_t)b * hw * F;
    const float* viewb = view + (size_t)b * hw * F;
    const int CO = (MODE == 0) ? 2 * F : F;
    float4 r = make_float4(0.f, 0.f, 0.f, 0.f);
    if (!WARP_REF && MODE != 1) r = __ldg(reinterpret_cast<const float4*>(refb + (size_t)pix * F + g * 4));
    const int d0 = blockIdx.y * K1_DCHUNK;
    const int d1 = min(D, d0 + K1_DCHUNK);
    for (int d = d0; d < d1; ++d) {
        const float* H = hv + ((size_t)b * D + d) * 9;
        float u, v;
        homography_uv(H, x, y, u, v);
        const Sample s = make_sample(u, v, h, w);
        float4 wv = sample4(s, viewb, w, F, g * 4);
        if (WARP_REF && MODE != 1) {
            float ur, vr;
            homography_uv(hr + ((size_t)b * D + d) * 9, x, y, ur, vr);
            const Sample sr = make_sample(ur, vr, h, w);
            r = sample4(sr, refb, w, F, g * 4);
        }
        OutT* o = out + (((size_t)b * D + d) * hw + pix) * CO;
        if (MODE == 0) {
            store4(o + g * 4, r);
            store4(o + F + g * 4, wv);
        } else if (MODE == 1) {
            store4(o + g * 4, wv);
        } else {
            const float m = s.valid ? 1.0f : 0.0f;   // model.py:277-278
            wv.x = MUL(fabsf(SUB(wv.x, r.x)), m);
            wv.y = MUL(fabsf(SUB(wv.y, r.y)), m);
            wv.z = MUL(fabsf(SUB(wv.z, r.z)), m);
            wv.w = MUL(fabsf(SUB(wv.w, r.w)), m);
            store4(o + g * 4, wv);
        }
    }
}


// K1, shared-coordinate version (F/4 = G lanes per pixel, G a power of two <= 32).  The G lanes of a
// pixel need the SAME sample cell and weights for a plane, and the IEEE divisions of the homography
// are the expensive part of the kernel: each lane therefore evaluates the homography of a different
// plane of the 8-plane chunk (lane g -> planes g, g+G, ...), and the loop over planes fetches the
// cell index and the four area weights from the owning lane with width-G shuffles.
//   cell: y0*w + x0  |  -1 = outside (output exactly 0, homography_warping.py:39-43,97-99)  |  -2 = not finite
template <typename OutT>
__device__ __forceinline__ float blend_out(float wa, float wb, float wc, float wd, float a, float b, float c, float d) {
    if (sizeof(OutT) == 4) return ADD(ADD(ADD(MUL(wa, a), MUL(wb, b)), MUL(wc, c)), MUL(wd, d));   // oracle order
    return fmaf(wd, d, fmaf(wc, c, fmaf(wb, b, wa * a)));          // bf16 volume: rounding dominates
}

template <typename OutT, int MODE, int G>
__global__ void __launch_bounds__(256)
k_build_cost_volume(const float* __restrict__ ref, const float* __restrict__ view, const float* __restrict__ hv,
                    int D, int h, int w, OutT* __restrict__ out) {
    constexpr int F = 4 * G;
    constexpr int NS = (G >= K1_DCHUNK) ? 1 : K1_DCHUNK / G;      // samples evaluated per lane
    const int hw = h * w;
    // a block is a 2-D patch of 8 x (256/G/8) pixels: neighbouring rows share their bilinear corner
    // rows in L1 instead of re-fetching them from L2
    constexpr int PPB = 256 / G, PH = (PPB >= 8) ? PPB / 8 : 1, PW = PPB / PH;
    const int ptx = (w + PW - 1) / PW;
    const int pl = threadIdx.x / G, g = threadIdx.x % G;
    const int x = (blockIdx.x % ptx) * PW + pl % PW, y = (blockIdx.x / ptx) * PH + pl / PW;
    const bool live = x < w && y < h;
    const int pix = live ? y * w + x : hw - 1;
    const int b = blockIdx.z;
    const float* viewb = view + (size_t)b * hw * F;
    constexpr int CO = (MODE == 0) ? 2 * F : F;
    float4 r = make_float4(0.f, 0.f, 0.f, 0.f);
    if (MODE != 1) r = __ldg(reinterpret_cast<const float4*>(ref + ((size_t)b * hw + pix) * F + g * 4));
    const int d0 = blockIdx.y * K1_DCHUNK;
    int cell[NS];
    float wa[NS], wb[NS], wc[NS], wd[NS];
#pragma unroll
    for (int k = 0; k < NS; ++k) {
        const int d = d0 + g + k * G;
        cell[k] = -1;
        wa[k] = wb[k] = wc[k] = wd[k] = 0.f;
        if (g + k * G < K1_DCHUNK && d < D) {
            float u, v;
            homography_uv(hv + ((size_t)b * D + d) * 9, x, y, u, v);
            const Sample s = make_sample(u, v, h, w);
            cell[k] = s.valid ? s.y0 * w + s.x0 : (s.finite ? -1 : -2);
            wa[k] = s.wa; wb[k] = s.wb; wc[k] = s.wc; wd[k] = s.wd;
        }
    }
    OutT* o = out + (((size_t)b * D + d0) * hw + pix) * CO + g * 4;
    const size_t ostride = (size_t)hw * CO;
#pragma unroll
    for (int j = 0; j < K1_DCHUNK; ++j) {
        const int k = (G >= K1_DCHUNK) ? 0 : j / G;
        const int src = j % G;
        const int c = __shfl_sync(0xffffffffu, cell[k], src, G);
        const float a0 = __shfl_sync(0xffffffffu, wa[k], src, G), a1 = __shfl_sync(0xffffffffu, wb[k], src, G);
        const float a2 = __shfl_sync(0xffffffffu, wc[k], src, G), a3 = __shfl_sync(0xffffffffu, wd[k], src, G);
        if (d0 + j >= D) break;
        float4 wv;
        if (c >= 0) {
            const float* p = viewb + (size_t)c * F + g * 4;
            const float4 A = __ldg(reinterpret_cast<const float4*>(p));
            const float4 Bq = __ldg(reinterpret_cast<const float4*>(p + F));
            const float4 C = __ldg(reinterpret_cast<const float4*>(p + (size_t)w * F));
            const float4 Dq = __ldg(reinterpret_cast<const float4*>(p + (size_t)w * F + F));
            wv = make_float4(blend_out<OutT>(a0, a1, a2, a3, A.x, Bq.x, C.x, Dq.x), blend_out<OutT>(a0, a1, a2, a3, A.y, Bq.y, C.y, Dq.y),
                             blend_out<OutT>(a0, a1, a2, a3, A.z, Bq.z, C.z, Dq.z), blend_out<OutT>(a0, a1, a2, a3, A.w, Bq.w, C.w, Dq.w));
        } else {
            const float z = (c == -1) ? 0.0f : __int_as_float(0x7fc00000);
            wv = make_float4(z, z, z, z);
        }
        if (!live) continue;
        OutT* oj = o + (size_t)j * ostride;
        if (MODE == 0) {
            store4(oj, r);
            store4(oj + F, wv);
        } else if (MODE == 1) {
            store4(oj, wv);
        } else {
            const float m = (c >= 0) ? 1.0f : 0.0f;   // model.py:277-278
            wv.x = MUL(fabsf(SUB(wv.x, r.x)), m);
            wv.y = MUL(fabsf(SUB(wv.y, r.y)), m);
            wv.z = MUL(fabsf(SUB(wv.z, r.z)), m);
            wv.w = MUL(fabsf(SUB(wv.w, r.w)), m);
            store4(oj, wv);
        }
    }
}


// K1 for bf16 cost volumes: the source feature map is first rounded to bf16 (one tiny pass; the
// volume it feeds is bf16 anyway), so that a bilinear corner of 8 channels is ONE 16-byte load and a
// pixel needs F/8 lanes: half the L1 wavefronts, shuffles and instructions per output byte of the
// fp32-source kernel, and 16-byte streaming stores.  Same sample sharing scheme (lane g evaluates the
// homography of planes g, g+G8, ... of the 8-plane chunk).
template <bool F16>
__device__ __forceinline__ void unpack8(const uint4 u, float* f) {
    if (F16) {
        const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&u.x)), b = __half22float2(*reinterpret_cast<const __half2*>(&u.y));
        const float2 c = __half22float2(*reinterpret_cast<const __half2*>(&u.z)), d = __half22float2(*reinterpret_cast<const __half2*>(&u.w));
        f[0] = a.x; f[1] = a.y; f[2] = b.x; f[3] = b.y; f[4] = c.x; f[5] = c.y; f[6] = d.x; f[7] = d.y;
        return;
    }
    // bf16 -> fp32 is a 16-bit shift: one SHL for the low half, one AND for the high half
    f[0] = __uint_as_float(u.x << 16); f[1] = __uint_as_float(u.x & 0xffff0000u);
    f[2] = __uint_as_float(u.y << 16); f[3] = __uint_as_float(u.y & 0xffff0000u);
    f[4] = __uint_as_float(u.z << 16); f[5] = __uint_as_float(u.z & 0xffff0000u);
    f[6] = __uint_as_float(u.w << 16); f[7] = __uint_as_float(u.w & 0xffff0000u);
}
template <bool F16>
__device__ __forceinline__ uint4 pack8(const float* f) {
    if (F16) {
        uint4 u;
        u.x = f16x2_sat(f[0], f[1]); u.y = f16x2_sat(f[2], f[3]); u.z = f16x2_sat(f[4], f[5]); u.w = f16x2_sat(f[6], f[7]);
        return u;
    }
    __nv_bfloat162 a = __floats2bfloat162_rn(f[0], f[1]), b = __floats2bfloat162_rn(f[2], f[3]);
    __nv_bfloat162 c = __floats2bfloat162_rn(f[4], f[5]), d = __floats2bfloat162_rn(f[6], f[7]);
    uint4 u;
    u.x = *reinterpret_cast<unsigned*>(&a); u.y = *reinterpret_cast<unsigned*>(&b);
    u.z = *reinterpret_cast<unsigned*>(&c); u.w = *reinterpret_cast<unsigned*>(&d);
    return u;
}

// packed-half blend of one channel pair: wa*a + wb*b + wc*c + wd*d in fp16 arithmetic (3 fused roundings).  The
// fp16 volume path only: its result is rounded to fp16 right after anyway, and the depth-MAE budget barely moves
// (2.6e-4 -> 2.9e-4 of the range in tests/precision_emulation.py) while the kernel drops from 17 to 4 instructions per
// channel pair and leaves the instruction-issue limit for the HBM one.
__device__ __forceinline__ unsigned hblend2(unsigned a, unsigned b, unsigned c, unsigned d, __half2 wa, __half2 wb, __half2 wc,
                                            __half2 wd) {
    __half2 r = __hmul2(wa, *reinterpret_cast<const __half2*>(&a));
    r = __hfma2(wb, *reinterpret_cast<const __half2*>(&b), r);
    r = __hfma2(wc, *reinterpret_cast<const __half2*>(&c), r);
    r = __hfma2(wd, *reinterpret_cast<const __half2*>(&d), r);
    return *reinterpret_cast<unsigned*>(&r);
}

template <int MODE, int G8, bool F16>
__global__ void __launch_bounds__(256)
k_build_cost_volume_h(const float* __restrict__ ref, const uint16_t* __restrict__ view, const float* __restrict__ hv,
                      int D, int h, int w, uint16_t* __restrict__ out) {
    constexpr int F = 8 * G8;
    constexpr int NS = (G8 >= K1_DCHUNK) ? 1 : K1_DCHUNK / G8;
    const int hw = h * w;
    // a block is a 2-D patch of 8 x (256/G8/8) pixels (vertical reuse of the corner rows in L1)
    constexpr int PPB = 256 / G8, PH = (PPB >= 8) ? PPB / 8 : 1, PW = PPB / PH;
    const int ptx = (w + PW - 1) / PW;
    const int pl = threadIdx.x / G8, g = threadIdx.x % G8;
    const int x = (blockIdx.x % ptx) * PW + pl % PW, y = (blockIdx.x / ptx) * PH + pl / PW;
    const bool live = x < w && y < h;
    const int pix = live ? y * w + x : hw - 1;
    const int b = blockIdx.z;
    const uint16_t* viewb = view + (size_t)b * hw * F;
    constexpr int CO = (MODE == 0) ? 2 * F : F;
    float r[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) r[i] = 0.f;
    if (MODE != 1) {
        const float4 r0 = __ldg(reinterpret_cast<const float4*>(ref + ((size_t)b * hw + pix) * F + g * 8));
        const float4 r1 = __ldg(reinterpret_cast<const float4*>(ref + ((size_t)b * hw + pix) * F + g * 8 + 4));
        r[0] = r0.x; r[1] = r0.y; r[2] = r0.z; r[3] = r0.w; r[4] = r1.x; r[5] = r1.y; r[6] = r1.z; r[7] = r1.w;
    }
    const int d0 = blockIdx.y * K1_DCHUNK;
    // cell: y0*w + x0, or -1 when the sample is outside (weights 0 -> output exactly 0) / not finite
    // (weights NaN -> output NaN, as the reference's arithmetic would give): the plane loop is branch-free
    int cell[NS];
    float wa[NS], wb[NS], wc[NS], wd[NS];
#pragma unroll
    for (int k = 0; k < NS; ++k) {
        const int d = d0 + g + k * G8;
        cell[k] = -1;
        wa[k] = wb[k] = wc[k] = wd[k] = 0.f;
        if (g + k * G8 < K1_DCHUNK && d < D) {
            float u, v;
            homography_uv(hv + ((size_t)b * D + d) * 9, x, y, u, v);
            const Sample s = make_sample(u, v, h, w);
            cell[k] = s.valid ? s.y0 * w + s.x0 : -1;
            const float bad = s.finite ? 0.f : __int_as_float(0x7fc00000);
            wa[k] = s.valid ? s.wa : bad; wb[k] = s.valid ? s.wb : bad;
            wc[k] = s.valid ? s.wc : bad; wd[k] = s.valid ? s.wd : bad;
        }
    }
    const uint16_t* vbase = viewb + g * 8;
    const int rowpitch = w * F;
    uint16_t* oj = out + (((size_t)b * D + d0) * hw + pix) * CO + g * 8;
    const size_t ostride = (size_t)hw * CO;
    const uint4 rpk = pack8<F16>(r);
#pragma unroll
    for (int j = 0; j < K1_DCHUNK; ++j, oj += ostride) {
        const int k = (G8 >= K1_DCHUNK) ? 0 : j / G8;
        const int src = j % G8;
        const int c = __shfl_sync(0xffffffffu, cell[k], src, G8);
        const float a0 = __shfl_sync(0xffffffffu, wa[k], src, G8), a1 = __shfl_sync(0xffffffffu, wb[k], src, G8);
        const float a2 = __shfl_sync(0xffffffffu, wc[k], src, G8), a3 = __shfl_sync(0xffffffffu, wd[k], src, G8);
        if (d0 + j >= D) break;
        const uint16_t* p = vbase + (ptrdiff_t)max(c, 0) * F;
        if (F16 && MODE != 2) {
            const uint4 ua = __ldg(reinterpret_cast<const uint4*>(p)), ub = __ldg(reinterpret_cast<const uint4*>(p + F));
            const uint4 uc = __ldg(reinterpret_cast<const uint4*>(p + rowpitch));
            const uint4 ud = __ldg(reinterpret_cast<const uint4*>(p + rowpitch + F));
            const __half2 h0 = __float2half2_rn(a0), h1 = __float2half2_rn(a1), h2 = __float2half2_rn(a2), h3 = __float2half2_rn(a3);
            uint4 o;
            o.x = hblend2(ua.x, ub.x, uc.x, ud.x, h0, h1, h2, h3);
            o.y = hblend2(ua.y, ub.y, uc.y, ud.y, h0, h1, h2, h3);
            o.z = hblend2(ua.z, ub.z, uc.z, ud.z, h0, h1, h2, h3);
            o.w = hblend2(ua.w, ub.w, uc.w, ud.w, h0, h1, h2, h3);
            if (!live) continue;
            if (MODE == 0) {
                __stcs(reinterpret_cast<uint4*>(oj), rpk);
                __stcs(reinterpret_cast<uint4*>(oj + F), o);
            } else {
                __stcs(reinterpret_cast<uint4*>(oj), o);
            }
            continue;
        }
        float A[8], Bq[8], C[8], Dq[8], wv[8];
        unpack8<F16>(__ldg(reinterpret_cast<const uint4*>(p)), A);
        unpack8<F16>(__ldg(reinterpret_cast<const uint4*>(p + F)), Bq);
        unpack8<F16>(__ldg(reinterpret_cast<const uint4*>(p + rowpitch)), C);
        unpack8<F16>(__ldg(reinterpret_cast<const uint4*>(p + rowpitch + F)), Dq);
#pragma unroll
        for (int i = 0; i < 8; ++i) wv[i] = fmaf(a3, Dq[i], fmaf(a2, C[i], fmaf(a1, Bq[i], a0 * A[i])));
        if (!live) continue;
        if (MODE == 0) {
            __stcs(reinterpret_cast<uint4*>(oj), rpk);
            __stcs(reinterpret_cast<uint4*>(oj + F), pack8<F16>(wv));
        } else if (MODE == 1) {
            __stcs(reinterpret_cast<uint4*>(oj), pack8<F16>(wv));
        } else {
            const float m = (c >= 0) ? 1.0f : 0.0f;   // model.py:277-278
#pragma unroll
            for (int i = 0; i < 8; ++i) wv[i] = fabsf(wv[i] - r[i]) * m;
            __stcs(reinterpret_cast<uint4*>(oj), pack8<F16>(wv));
        }
    }
}

template <bool F16>
__global__ void k_f32_to_16(const float* __restrict__ s, uint16_t* __restrict__ d, long long n4) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
        const float4 v = __ldg(reinterpret_cast<const float4*>(s) + i);
        uint2 pk;
        if (F16) {
            pk.x = f16x2_sat(v.x, v.y);
            pk.y = f16x2_sat(v.z, v.w);
        } else {
            __nv_bfloat162 lo = __floats2bfloat162_rn(v.x, v.y), hi = __floats2bfloat162_rn(v.z, v.w);
            pk.x = *reinterpret_cast<unsigned*>(&lo);
            pk.y = *reinterpret_cast<unsigned*>(&hi);
        }
        reinterpret_cast<uint2*>(d)[i] = pk;
    }
}

// ------------------------------------------------------------------ soft-argmin (K4)
// one thread = one output pixel; single pass over D with an online softmax; the x4 variant
// interpolates the logits on the fly (tf.image.resize_images, align_corners=True).
template <int UP>
__global__ void __launch_bounds__(256)
k_prob2depth(const float* __restrict__ vol, int B, int D, int H, int W, const float* __restrict__ dstart,
             const float* __restrict__ dint, float* __restrict__ depth, float* __restrict__ prob) {
    const int Ho = H * UP, Wo = W * UP;
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (long long)B * Ho * Wo) return;
    const int X = (int)(idx % Wo), Y = (int)((idx / Wo) % Ho), b = (int)(idx / ((long long)Wo * Ho));
    const size_t plane = (size_t)H * W;
    const float* vb = vol + (size_t)b * D * plane;
    int x0 = X, x1 = X, y0 = Y, y1 = Y;
    float fx = 0.f, fy = 0.f;
    if (UP > 1) {
        const float sy = DIV((float)(H - 1), (float)(Ho - 1)), sx = DIV((float)(W - 1), (float)(Wo - 1));
        const float srcy = MUL((float)Y, sy), srcx = MUL((float)X, sx);
        y0 = (int)floorf(srcy);
        x0 = (int)floorf(srcx);
        y1 = min(y0 + 1, H - 1);
        x1 = min(x0 + 1, W - 1);
        fy = SUB(srcy, (float)y0);
        fx = SUB(srcx, (float)x0);
    }
    const size_t o00 = (size_t)y0 * W + x0, o01 = (size_t)y0 * W + x1, o10 = (size_t)y1 * W + x0,
                 o11 = (size_t)y1 * W + x1;
    auto logit = [&](int d) -> float {
        const float* p = vb + (size_t)d * plane;
        if (UP == 1) return __ldg(p + o00);
        const float tl = __ldg(p + o00), tr = __ldg(p + o01), bl = __ldg(p + o10), br = __ldg(p + o11);
        const float top = ADD(tl, MUL(SUB(tr, tl), fx));
        const float bot = ADD(bl, MUL(SUB(br, bl), fx));
        return ADD(top, MUL(SUB(bot, top), fy));
    };
    const float ds = dstart[b], di = dint[b];
    const float de = ADD(ds, MUL(SUB((float)D, 1.0f), di));
    const float step = DIV(SUB(de, ds), (float)max(D - 1, 1));
    float m = -INFINITY, s = 0.f, ws = 0.f;
    for (int d = 0; d < D; ++d) {
        const float t = -logit(d);
        if (t > m) {
            const float sc = expf(m - t);
            s *= sc;
            ws *= sc;
            m = t;
        }
        const float e = expf(t - m);
        s += e;
        ws += ADD(ds, MUL((float)d, step)) * e;
    }
    const float est = ws / s;
    depth[idx] = est;
    if (prob) {
        const float t = DIV(SUB(est, ds), di);
        const int l0 = min(max((int)floorf(t), 0), D - 1);
        const int l1 = min(max(l0 - 1, 0), D - 1);
        const int r0 = min(max((int)ceilf(t), 0), D - 1);
        const int r1 = min(max(r0 + 1, 0), D - 1);
        const float inv = 1.0f / s;
        float p = expf(-logit(l0) - m) * inv;
        p += expf(-logit(l1) - m) * inv;
        p += expf(-logit(r0) - m) * inv;
        p += expf(-logit(r1) - m) * inv;
        prob[idx] = p;
    }
}


// K4 at the volume's own resolution: a block is 8 depth slices (warps) x 32 lanes, a lane owns VEC
// consecutive pixels (VEC = 4: 16-byte plane reads).  Every slice runs an online softmax over its planes
// d = slice, slice+8, ... in batches of 4 planes (4 independent loads in flight, ONE rescale of the
// running sums per batch); the 8 partial (max, sum, weighted sum) triples are merged through shared memory.
constexpr int K4_SLICES = 8;
constexpr float K4_LOG2E = 1.4426950408889634f;

template <int VEC>
__global__ void __launch_bounds__(256)
k_prob2depth_sliced(const float* __restrict__ vol, int B, int D, long long plane, const float* __restrict__ dstart,
                    const float* __restrict__ dint, float* __restrict__ depth, float* __restrict__ prob) {
    __shared__ float sm_m[K4_SLICES][32 * VEC], sm_s[K4_SLICES][32 * VEC], sm_w[K4_SLICES][32 * VEC];
    const int lane = threadIdx.x & 31, slice = threadIdx.x >> 5;
    const long long total = (long long)B * plane;                 // VEC == 4 requires plane % 4 == 0
    const long long idx = ((long long)blockIdx.x * 32 + lane) * VEC;
    const bool live = idx < total;
    const long long pidx = live ? idx : total - VEC;
    const int b = (int)(pidx / plane);
    const float* vb = vol + (size_t)b * D * plane + (size_t)(pidx - (long long)b * plane);
    const float ds = dstart[b], di = dint[b];
    const float de = ADD(ds, MUL(SUB((float)D, 1.0f), di));
    const float step = DIV(SUB(de, ds), (float)max(D - 1, 1));
    float m[VEC], s[VEC], ws[VEC];
#pragma unroll
    for (int v = 0; v < VEC; ++v) { m[v] = -INFINITY; s[v] = 0.f; ws[v] = 0.f; }
    for (int d = slice; d < D; d += 4 * K4_SLICES) {
        float t[4][VEC];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int dq = d + q * K4_SLICES;
            if (dq < D) {
                if (VEC == 4) {
                    const float4 r = __ldcs(reinterpret_cast<const float4*>(vb + (size_t)dq * plane));
                    t[q][0] = -r.x; t[q][1 % VEC] = -r.y; t[q][2 % VEC] = -r.z; t[q][3 % VEC] = -r.w;
                } else {
                    t[q][0] = -__ldcs(vb + (size_t)dq * plane);
                }
            } else {
#pragma unroll
                for (int v = 0; v < VEC; ++v) t[q][v] = -INFINITY;
            }
        }
#pragma unroll
        for (int v = 0; v < VEC; ++v) {
            const float mn = fmaxf(fmaxf(fmaxf(t[0][v], t[1][v]), fmaxf(t[2][v], t[3][v])), m[v]);
            const float sc = exp2f((m[v] - mn) * K4_LOG2E);        // m = -inf at the start: exp2(-inf) = 0
            float sa = s[v] * sc, wa = ws[v] * sc;
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const float e = exp2f((t[q][v] - mn) * K4_LOG2E);  // padded planes: exp2(-inf) = 0
                sa += e;
                wa = fmaf(ADD(ds, MUL((float)(d + q * K4_SLICES), step)), e, wa);
            }
            m[v] = mn; s[v] = sa; ws[v] = wa;
        }
    }
#pragma unroll
    for (int v = 0; v < VEC; ++v) {
        sm_m[slice][lane * VEC + v] = m[v];
        sm_s[slice][lane * VEC + v] = s[v];
        sm_w[slice][lane * VEC + v] = ws[v];
    }
    __syncthreads();
    // 32*VEC pixels of the block are finalised by the first 32*VEC threads
    const int pl = threadIdx.x;
    if (pl >= 32 * VEC) return;
    const long long oidx = (long long)blockIdx.x * 32 * VEC + pl;
    if (oidx >= total) return;
    float M = -INFINITY;
#pragma unroll
    for (int k = 0; k < K4_SLICES; ++k) M = fmaxf(M, sm_m[k][pl]);
    float S = 0.f, WS = 0.f;
#pragma unroll
    for (int k = 0; k < K4_SLICES; ++k) {
        const float mk = sm_m[k][pl];
        if (mk == -INFINITY) continue;                     // slice without planes (D < 8)
        const float sc = exp2f((mk - M) * K4_LOG2E);
        S = fmaf(sm_s[k][pl], sc, S);
        WS = fmaf(sm_w[k][pl], sc, WS);
    }
    const float est = WS / S;
    depth[oidx] = est;
    if (prob) {
        const int ob = (int)(oidx / plane);
        const float* vo = vol + (size_t)ob * D * plane + (size_t)(oidx - (long long)ob * plane);
        const float dso = dstart[ob], dio = dint[ob];
        const float t = DIV(SUB(est, dso), dio);
        const int l0 = min(max((int)floorf(t), 0), D - 1);
        const int l1 = min(max(l0 - 1, 0), D - 1);
        const int r0 = min(max((int)ceilf(t), 0), D - 1);
        const int r1 = min(max(r0 + 1, 0), D - 1);
        const float inv = 1.0f / S;
        float pr = expf(-__ldg(vo + (size_t)l0 * plane) - M) * inv;
        pr += expf(-__ldg(vo + (size_t)l1 * plane) - M) * inv;
        pr += expf(-__ldg(vo + (size_t)r0 * plane) - M) * inv;
        pr += expf(-__ldg(vo + (size_t)r1 * plane) - M) * inv;
        prob[oidx] = pr;
    }
}

// 2^x on the SFU (MUFU.EX2, ~2 ulp, denormal results flushed): the soft-argmin weights are >= 2^-126 or irrelevant
__device__ __forceinline__ float ex2_approx(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

// K4 fused with the x4 logit upsampling (model.py:68-76 + :80-109).  The kernel is instruction bound (D*16*h*w
// interpolations + exponentials against 4*D*h*w bytes), so it is organised to minimise instructions per output:
//   block  : 8 depth slices (warps) x 32 lanes, one output row Y; lane k owns the 4 output pixels X = 4k..4k+3
//   texels : those 4 pixels read source columns {k-1, k, k+1} only (x0 = floor(X*(W-1)/(4W-1)) is k-1 or k), so a
//            plane costs 6 loads per lane (3 columns x 2 rows) instead of 16; 4 planes = 24 loads in flight
//   softmax: batched online softmax per output (ONE rescale per 4 planes), slices merged through shared memory
// TF's lerp order (top = tl + (tr-tl)*fx, bot likewise, top + (bot-top)*fy) is kept, each "a + b*c" as one FMA.
template <int UP>
__global__ void __launch_bounds__(256)
k_prob2depth_up_sliced(const float* __restrict__ vol, int B, int D, int H, int W, const float* __restrict__ dstart,
                       const float* __restrict__ dint, float* __restrict__ depth, float* __restrict__ prob) {
    static_assert(UP == 4, "column ownership is derived for x4");
    __shared__ float sm_m[K4_SLICES][128], sm_s[K4_SLICES][128], sm_w[K4_SLICES][128];
    const int lane = threadIdx.x & 31, slice = threadIdx.x >> 5;
    const int Ho = H * UP, Wo = W * UP;
    const int xb = (W + 31) / 32;
    const int bx = blockIdx.x % xb;
    const int Y = (blockIdx.x / xb) % Ho, b = blockIdx.x / (xb * Ho);
    const int k = min(bx * 32 + lane, W - 1);
    const size_t plane = (size_t)H * W;
    const float* vb = vol + (size_t)b * D * plane;
    const float sy = DIV((float)(H - 1), (float)(Ho - 1)), sx = DIV((float)(W - 1), (float)(Wo - 1));
    const float srcy = MUL((float)Y, sy);
    const int y0 = (int)floorf(srcy);
    const int y1 = min(y0 + 1, H - 1);
    const float fy = SUB(srcy, (float)y0);
    float fx[4];
    bool hi[4];                       // x0 == k (else k-1)
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const float srcx = MUL((float)(4 * k + j), sx);
        const int x0 = (int)floorf(srcx);
        fx[j] = SUB(srcx, (float)x0);
        hi[j] = x0 >= k;
    }
    const int c0 = max(k - 1, 0), c2 = min(k + 1, W - 1);
    const float* r0 = vb + (size_t)y0 * W + (size_t)slice * plane;
    const float* r1 = vb + (size_t)y1 * W + (size_t)slice * plane;
    const size_t bstep = (size_t)K4_SLICES * plane;
    const float ds = dstart[b], di = dint[b];
    const float de = ADD(ds, MUL(SUB((float)D, 1.0f), di));
    const float step = DIV(SUB(de, ds), (float)max(D - 1, 1));
    float m[4], s[4], ws[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) { m[j] = -INFINITY; s[j] = 0.f; ws[j] = 0.f; }
    // one batch of 4 planes; FULL = all four planes exist (no per-plane predicates in the steady state)
    auto batch = [&](int d, auto full_tag) {
        constexpr bool FULL = decltype(full_tag)::value;
        float a[4][2][3];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const size_t off = (FULL || d + q * K4_SLICES < D) ? (size_t)q * bstep : 0;
            a[q][0][0] = __ldg(r0 + off + c0); a[q][0][1] = __ldg(r0 + off + k); a[q][0][2] = __ldg(r0 + off + c2);
            a[q][1][0] = __ldg(r1 + off + c0); a[q][1][1] = __ldg(r1 + off + k); a[q][1][2] = __ldg(r1 + off + c2);
        }
        float dep[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) dep[q] = ADD(ds, MUL((float)(d + q * K4_SLICES), step));
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            float t[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const float tl = hi[j] ? a[q][0][1] : a[q][0][0], tr = hi[j] ? a[q][0][2] : a[q][0][1];
                const float bl = hi[j] ? a[q][1][1] : a[q][1][0], br = hi[j] ? a[q][1][2] : a[q][1][1];
                const float top = fmaf(tr - tl, fx[j], tl), bot = fmaf(br - bl, fx[j], bl);
                const float v = fmaf(top - bot, fy, -top);                    // -(top + (bot - top) * fy)
                t[q] = (FULL || d + q * K4_SLICES < D) ? v : -INFINITY;
            }
            const float mn = fmaxf(fmaxf(fmaxf(t[0], t[1]), fmaxf(t[2], t[3])), m[j]);
            const float mnl = mn * K4_LOG2E;
            const float sc = ex2_approx(fmaf(m[j], K4_LOG2E, -mnl));          // m = -inf at the start: 2^-inf = 0
            float sa = s[j] * sc, wa = ws[j] * sc;
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const float e = ex2_approx(fmaf(t[q], K4_LOG2E, -mnl));
                sa += e;
                wa = fmaf(dep[q], e, wa);
            }
            m[j] = mn; s[j] = sa; ws[j] = wa;
        }
    };
    for (int d = slice; d < D; d += 4 * K4_SLICES, r0 += 4 * bstep, r1 += 4 * bstep) {
        if (d + 3 * K4_SLICES < D) batch(d, std::true_type());
        else batch(d, std::false_type());
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        sm_m[slice][lane * 4 + j] = m[j]; sm_s[slice][lane * 4 + j] = s[j]; sm_w[slice][lane * 4 + j] = ws[j];
    }
    __syncthreads();
    const int pl = threadIdx.x;
    const int X = bx * 128 + pl;
    if (pl >= 128 || X >= Wo) return;
    float M = -INFINITY;
#pragma unroll
    for (int q = 0; q < K4_SLICES; ++q) M = fmaxf(M, sm_m[q][pl]);
    float S = 0.f, WS = 0.f;
#pragma unroll
    for (int q = 0; q < K4_SLICES; ++q) {
        const float mk = sm_m[q][pl];
        if (mk == -INFINITY) continue;                     // slice without planes (D < 8)
        const float sc = exp2f((mk - M) * K4_LOG2E);
        S = fmaf(sm_s[q][pl], sc, S);
        WS = fmaf(sm_w[q][pl], sc, WS);
    }
    const float est = WS / S;
    const size_t oidx = ((size_t)b * Ho + Y) * Wo + X;
    depth[oidx] = est;
    if (prob) {
        const float srcx = MUL((float)X, sx);
        const int x0 = (int)floorf(srcx), x1 = min(x0 + 1, W - 1);
        const float gx = SUB(srcx, (float)x0);
        const float t = DIV(SUB(est, ds), di);
        const int l0 = min(max((int)floorf(t), 0), D - 1);
        const int l1 = min(max(l0 - 1, 0), D - 1);
        const int q0 = min(max((int)ceilf(t), 0), D - 1);
        const int q1 = min(max(q0 + 1, 0), D - 1);
        const float inv = 1.0f / S;
        auto logit = [&](int d) -> float {
            const float* p0 = vb + (size_t)d * plane + (size_t)y0 * W;
            const float* p1 = vb + (size_t)d * plane + (size_t)y1 * W;
            const float tl = __ldg(p0 + x0), tr = __ldg(p0 + x1), bl = __ldg(p1 + x0), br = __ldg(p1 + x1);
            const float top = fmaf(tr - tl, gx, tl), bot = fmaf(br - bl, gx, bl);
            return fmaf(bot - top, fy, top);
        };
        float pr = expf(-logit(l0) - M) * inv;
        pr += expf(-logit(l1) - M) * inv;
        pr += expf(-logit(q0) - M) * inv;
        pr += expf(-logit(q1) - M) * inv;
        prob[oidx] = pr;
    }
}

// ------------------------------------------------------------------ refinement stage geometry (SURVEY.md 8(f) N2)
// transform_depth, homography_warping.py:275-326: depth of the LEFT view re-expressed in the RIGHT camera, on the
// left pixel grid.  mv = (mat (9), vec (3)) from k_bydepth_setup(left, right).  The reference's clip upper bounds
// (tf.reduce_max of the clipped tensor itself) never bind.
__global__ void k_transform_depth(const float* __restrict__ depth, const float* __restrict__ mv, int B, int H, int W,
                                  int inverse_depth, float* __restrict__ out) {
    const long long n = (long long)B * H * W;
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int x = (int)(i % W), y = (int)((i / W) % H), b = (int)(i / ((long long)W * H));
    const float* m = mv + (size_t)b * 12;
    float d = depth[i];
    const bool valid = d > 1e-10f;
    if (inverse_depth) {
        d = fmaxf(d, 1e-10f);
        d = DIV(1.0f, d);
        d = MUL(d, valid ? 1.0f : 0.0f);
    }
    const float px = MUL(ADD((float)x, 0.5f), d), py = MUL(ADD((float)y, 0.5f), d);
    float z = ADD(ADD(ADD(MUL(m[6], px), MUL(m[7], py)), MUL(m[8], d)), m[11]);
    if (inverse_depth) {
        z = fmaxf(z, 1e-10f);
        z = DIV(1.0f, z);
        z = MUL(z, valid ? 1.0f : 0.0f);
    }
    out[i] = z;
}

// geo_group of model.py:286-326, 328-337 in one pass: (B,D,H,W,1+C+2) =
//   [ |d_ref - v| / di / D | (|warp(d_view_t, H_d) - v| / di / D) * mask, repeated C times (the reference tiles the mask to
//     the C feature channels, SURVEY H7) | |wg - d_ref| * wg_mask | d_ref ],   v = start + d * interval
__global__ void __launch_bounds__(256)
k_refine_geo_group(const float* __restrict__ d_ref, const float* __restrict__ d_view_t, const float* __restrict__ hv,
                   const float* __restrict__ wg, const uint8_t* __restrict__ wg_mask, const float* __restrict__ dstart,
                   const float* __restrict__ dint, int B, int D, int H, int W, int C, float* __restrict__ out) {
    const long long n = (long long)B * D * H * W;
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int x = (int)(i % W), y = (int)((i / W) % H);
    const int d = (int)((i / ((long long)W * H)) % D), b = (int)(i / ((long long)W * H * D));
    const size_t pix = ((size_t)b * H + y) * W + x;
    const float ds = dstart[b], di = dint[b];
    const float val = ADD(ds, MUL((float)d, di));
    const float dr = d_ref[pix];
    const float g_ref = DIV(DIV(fabsf(SUB(dr, val)), di), (float)D);
    float u, v;
    homography_uv(hv + ((size_t)b * D + d) * 9, x, y, u, v);
    const Sample sm = make_sample(u, v, H, W);
    const float wd = sample1(sm, d_view_t + (size_t)b * H * W, W, 1, 0);
    const float g_view = MUL(DIV(DIV(fabsf(SUB(wd, val)), di), (float)D), sm.valid ? 1.0f : 0.0f);
    const float g_err = MUL(fabsf(SUB(wg[pix], dr)), wg_mask[pix] ? 1.0f : 0.0f);
    float* o = out + (size_t)i * (C + 3);
    o[0] = g_ref;
    for (int c = 0; c < C; ++c) o[1 + c] = g_view;
    o[C + 1] = g_err;
    o[C + 2] = dr;
}

// photo_group of model.py:269-281, 309-312, 328-336: (B,D,H,W,3C) = [L1 cost volume | |wf - ref_f| * mask | ref_f]
__global__ void __launch_bounds__(256)
k_refine_photo_group(const float* __restrict__ cost_photo, const float* __restrict__ wf, const uint8_t* __restrict__ mask,
                     const float* __restrict__ ref_f, long long nvox, long long plane, int C, float* __restrict__ out) {
    const long long n = nvox * C;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const long long vox = i / C;
        const int c = (int)(i % C);
        const long long b = vox / plane;                       // plane = D*H*W, pixels per batch element = H*W
        (void)b;
        out[vox * 3 * C + c] = cost_photo[i];
    }
}

__global__ void __launch_bounds__(256)
k_refine_photo_tail(const float* __restrict__ wf, const uint8_t* __restrict__ mask, const float* __restrict__ ref_f, int B,
                    int D, long long hw, int C, float* __restrict__ out) {
    const long long n = (long long)B * D * hw * C;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const int c = (int)(i % C);
        const long long vox = i / C;
        const long long p = vox % hw;
        const long long b = vox / (hw * D);
        const size_t pix = (size_t)b * hw + p;
        const float r = ref_f[pix * C + c];
        out[vox * 3 * C + C + c] = MUL(fabsf(SUB(wf[pix * C + c], r)), mask[pix] ? 1.0f : 0.0f);
        out[vox * 3 * C + 2 * C + c] = r;
    }
}

// get_visual_hull, homography_warping.py:329-387, for view_num = 2 (the only use: model.py:321-323 with num_depths = 2):
// (B,D,H,W,1) = ([ref > 0][ref beyond plane] + [w > 0][w beyond plane]) / 2, w = nearest warp of the transformed depth
__global__ void __launch_bounds__(256)
k_visual_hull2(const float* __restrict__ ref_depth, const float* __restrict__ trans, const float* __restrict__ hv,
               const float* __restrict__ dstart, const float* __restrict__ dint, int B, int D, int H, int W, int inverse_depth,
               float* __restrict__ out) {
    const long long n = (long long)B * D * H * W;
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int x = (int)(i % W), y = (int)((i / W) % H);
    const int d = (int)((i / ((long long)W * H)) % D), b = (int)(i / ((long long)W * H * D));
    const float val = ADD(dstart[b], MUL(dint[b], (float)d));
    const float r = ref_depth[((size_t)b * H + y) * W + x];
    float hull = (r > 0.0f && (inverse_depth ? r > val : val > r)) ? 1.0f : 0.0f;
    float u, v;
    homography_uv(hv + ((size_t)b * D + d) * 9, x, y, u, v);
    int x0, y0;
    bool valid;
    nearest_cell(u, v, H, W, x0, y0, valid);
    const float wd = trans[((size_t)b * H + y0) * W + x0];
    hull += (wd > 0.0f && (inverse_depth ? wd > val : val > wd)) ? 1.0f : 0.0f;
    out[i] = DIV(hull, 2.0f);
}

}  // namespace

// =========================================================================== C ABI
extern "C" int atvs_transform_depth(const float* depth, const float* left_cam, const float* right_cam, int B, int H, int W,
                                    int inverse_depth, float* out, atvs_stream_t stream) {
    ATVS_CHECK_ARG(depth && left_cam && right_cam && out, ATVS_E_NULL, "atvs_transform_depth: NULL pointer");
    ATVS_CHECK_ARG(B > 0 && H > 0 && W > 0, ATVS_E_SHAPE, "atvs_transform_depth: bad shape");
    cudaStream_t st = (cudaStream_t)stream;
    float* mv = nullptr;
    ATVS_CUDA(cudaMallocAsync(&mv, sizeof(float) * 12 * B, st));
    k_bydepth_setup<<<(B + 63) / 64, 64, 0, st>>>(left_cam, right_cam, B, mv);
    const long long n = (long long)B * H * W;
    k_transform_depth<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(depth, mv, B, H, W, inverse_depth, out);
    ATVS_CUDA(cudaFreeAsync(mv, st));
    ATVS_LAUNCH_CHECK();
    return 0;
}

extern "C" int atvs_refine_geo_group(const float* d_ref, const float* d_view_trans, const float* homographies, const float* wg,
                                     const uint8_t* wg_mask, const float* depth_start, const float* depth_interval, int B,
                                     int D, int H, int W, int C, float* out, atvs_stream_t stream) {
    ATVS_CHECK_ARG(d_ref && d_view_trans && homographies && wg && wg_mask && depth_start && depth_interval && out, ATVS_E_NULL,
                   "atvs_refine_geo_group: NULL pointer");
    ATVS_CHECK_ARG(B > 0 && D > 0 && H > 1 && W > 1 && C > 0, ATVS_E_SHAPE, "atvs_refine_geo_group: bad shape");
    const long long n = (long long)B * D * H * W;
    k_refine_geo_group<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(d_ref, d_view_trans, homographies, wg, wg_mask,
                                                                                   depth_start, depth_interval, B, D, H, W, C, out);
    ATVS_LAUNCH_CHECK();
    return 0;
}

extern "C" int atvs_refine_photo_group(const float* cost_photo, const float* warped_feature, const uint8_t* mask,
                                       const float* ref_feature, int B, int D, int H, int W, int C, float* out,
                                       atvs_stream_t stream) {
    ATVS_CHECK_ARG(cost_photo && warped_feature && mask && ref_feature && out, ATVS_E_NULL, "atvs_refine_photo_group: NULL pointer");
    ATVS_CHECK_ARG(B > 0 && D > 0 && H > 0 && W > 0 && C > 0, ATVS_E_SHAPE, "atvs_refine_photo_group: bad shape");
    const long long nvox = (long long)B * D * H * W;
    long long g = (nvox * C + 255) / 256;
    const long long cap = (long long)atvs_num_sms() * 8;
    if (g > cap) g = cap;
    cudaStream_t st = (cudaStream_t)stream;
    k_refine_photo_group<<<(unsigned)g, 256, 0, st>>>(cost_photo, warped_feature, mask, ref_feature, nvox, (long long)D * H * W, C, out);
    k_refine_photo_tail<<<(unsigned)g, 256, 0, st>>>(warped_feature, mask, ref_feature, B, D, (long long)H * W, C, out);
    ATVS_LAUNCH_CHECK();
    return 0;
}

extern "C" int atvs_visual_hull(const float* ref_depth, const float* trans_depth, const float* homographies,
                                const float* depth_start, const float* depth_interval, int B, int D, int H, int W,
                                int view_num, int inverse_depth, float* out, atvs_stream_t stream) {
    ATVS_CHECK_ARG(ref_depth && trans_depth && homographies && depth_start && depth_interval && out, ATVS_E_NULL,
                   "atvs_visual_hull: NULL pointer");
    ATVS_CHECK_ARG(B > 0 && D > 0 && H > 1 && W > 1, ATVS_E_SHAPE, "atvs_visual_hull: bad shape");
    ATVS_CHECK_ARG(view_num == 2, ATVS_E_UNSUP, "atvs_visual_hull: view_num=%d (the refinement stage uses 2)", view_num);
    const long long n = (long long)B * D * H * W;
    k_visual_hull2<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(ref_depth, trans_depth, homographies, depth_start,
                                                                               depth_interval, B, D, H, W, inverse_depth, out);
    ATVS_LAUNCH_CHECK();
    return 0;
}

extern "C" int atvs_get_homographies(const float* left_cam, const float* right_cam, int B, int D,
                                     const float* depth_start, const float* depth_interval, int inverse_depth,
                                     float* out, atvs_stream_t stream) {
    ATVS_CHECK_ARG(left_cam && right_cam && depth_start && depth_interval && out, ATVS_E_NULL,
                   "atvs_get_homographies: NULL pointer");
    ATVS_CHECK_ARG(B > 0 && D > 0, ATVS_E_SHAPE, "atvs_get_homographies: B=%d D=%d", B, D);
    const int n = B * D;
    k_get_homographies<<<(n + 127) / 128, 128, 0, (cudaStream_t)stream>>>(left_cam, right_cam, B, D, depth_start,
                                                                         depth_interval, inverse_depth, out);
    ATVS_LAUNCH_CHECK();
    return 0;
}

static int launch_warp(const float* image, const float* hm, const float* depth, int inverse_depth, bool bydepth,
                       int B, int H, int W, int C, int method, float* out, uint8_t* mask, cudaStream_t st) {
    const int vec = (C % 4 == 0) ? 4 : 1;
    const long long total = (long long)B * H * W * (C / vec);
    const unsigned grid = (unsigned)((total + 255) / 256);
    if (vec == 4) {
        if (bydepth) k_warp<4, true><<<grid, 256, 0, st>>>(image, hm, depth, inverse_depth, B, H, W, C, method, out, mask);
        else k_warp<4, false><<<grid, 256, 0, st>>>(image, hm, depth, inverse_depth, B, H, W, C, method, out, mask);
    } else {
        if (bydepth) k_warp<1, true><<<grid, 256, 0, st>>>(image, hm, depth, inverse_depth, B, H, W, C, method, out, mask);
        else k_warp<1, false><<<grid, 256, 0, st>>>(image, hm, depth, inverse_depth, B, H, W, C, method, out, mask);
    }
    ATVS_LAUNCH_CHECK();
    return 0;
}

extern "C" int atvs_homography_warping(const float* image, const float* homography, int B, int H, int W, int C,
                                       int method, float* out, uint8_t* mask, atvs_stream_t stream) {
    ATVS_CHECK_ARG(image && homography && out, ATVS_E_NULL, "atvs_homography_warping: NULL pointer");
    ATVS_CHECK_ARG(B > 0 && H > 1 && W > 1 && C > 0, ATVS_E_SHAPE, "atvs_homography_warping: bad shape %d %d %d %d", B,
                   H, W, C);
    ATVS_CHECK_ARG(method == 0 || method == 1, ATVS_E_UNSUP, "atvs_homography_warping: method %d", method);
    ATVS_CHECK_ARG(C % 4 != 0 || (((uintptr_t)image | (uintptr_t)out) & 15) == 0, ATVS_E_SHAPE,
                   "atvs_homography_warping: image/out must be 16-byte aligned");
    return launch_warp(image, homography, nullptr, 0, false, B, H, W, C, method, out, mask, (cudaStream_t)stream);
}

extern "C" int atvs_homography_warping_by_depth(const float* image, const float* left_cam, const float* right_cam,
                                                const float* depth_image, int B, int H, int W, int C, int method,
                                                int inverse_depth, float* out, uint8_t* mask, atvs_stream_t stream) {
    ATVS_CHECK_ARG(image && left_cam && right_cam && depth_image && out, ATVS_E_NULL,
                   "atvs_homography_warping_by_depth: NULL pointer");
    ATVS_CHECK_ARG(B > 0 && B <= 1024 && H > 1 && W > 1 && C > 0, ATVS_E_SHAPE,
                   "atvs_homography_warping_by_depth: bad shape");
    ATVS_CHECK_ARG(method == 0 || method == 1, ATVS_E_UNSUP, "atvs_homography_warping_by_depth: method %d", method);
    cudaStream_t st = (cudaStream_t)stream;
    float* mv = nullptr;
    ATVS_CUDA(cudaMallocAsync(&mv, sizeof(float) * 12 * B, st));
    k_bydepth_setup<<<(B + 63) / 64, 64, 0, st>>>(left_cam, right_cam, B, mv);
    ATVS_LAUNCH_CHECK();
    int rc = launch_warp(image, mv, depth_image, inverse_depth, true, B, H, W, C, method, out, mask, st);
    ATVS_CUDA(cudaFreeAsync(mv, st));
    return rc;
}

template <typename OutT, int G>
static void launch_k1_shared(const float* ref, const float* view, const float* hv, int D, int h, int w, int mode,
                             OutT* out, dim3 grid, cudaStream_t st) {
    if (mode == 0) k_build_cost_volume<OutT, 0, G><<<grid, 256, 0, st>>>(ref, view, hv, D, h, w, out);
    else if (mode == 1) k_build_cost_volume<OutT, 1, G><<<grid, 256, 0, st>>>(ref, view, hv, D, h, w, out);
    else k_build_cost_volume<OutT, 2, G><<<grid, 256, 0, st>>>(ref, view, hv, D, h, w, out);
}

template <typename OutT>
static int launch_k1(const float* ref, const float* view, const float* hv, const float* hr, int B, int D, int h, int w,
                     int F, int mode, OutT* out, cudaStream_t st) {
    const int G = F / 4;
    dim3 grid((unsigned)(((long long)h * w * G + 255) / 256), (unsigned)((D + K1_DCHUNK - 1) / K1_DCHUNK), (unsigned)B);
    if (!hr && (G == 1 || G == 2 || G == 4 || G == 8 || G == 16 || G == 32)) {
        const int ppb = 256 / G, ph = ppb >= 8 ? ppb / 8 : 1, pw = ppb / ph;
        grid.x = (unsigned)(((w + pw - 1) / pw) * ((h + ph - 1) / ph));
        switch (G) {
            case 1: launch_k1_shared<OutT, 1>(ref, view, hv, D, h, w, mode, out, grid, st); break;
            case 2: launch_k1_shared<OutT, 2>(ref, view, hv, D, h, w, mode, out, grid, st); break;
            case 4: launch_k1_shared<OutT, 4>(ref, view, hv, D, h, w, mode, out, grid, st); break;
            case 8: launch_k1_shared<OutT, 8>(ref, view, hv, D, h, w, mode, out, grid, st); break;
            case 16: launch_k1_shared<OutT, 16>(ref, view, hv, D, h, w, mode, out, grid, st); break;
            default: launch_k1_shared<OutT, 32>(ref, view, hv, D, h, w, mode, out, grid, st); break;
        }
        ATVS_LAUNCH_CHECK();
        return 0;
    }
#define K1_GO(MODE, WR) k_build_cost_volume_generic<OutT, MODE, WR><<<grid, 256, 0, st>>>(ref, view, hv, hr, D, h, w, F, out)
    if (hr) {
        if (mode == 0) K1_GO(0, true);
        else if (mode == 2) K1_GO(2, true);
        else K1_GO(1, false);
    } else {
        if (mode == 0) K1_GO(0, false);
        else if (mode == 1) K1_GO(1, false);
        else K1_GO(2, false);
    }
#undef K1_GO
    ATVS_LAUNCH_CHECK();
    return 0;
}

// 16-bit K1 (k_build_cost_volume_h): the source feature map is 16-bit in the volume's own format
static bool k1_h_supported(int F) { return F == 8 || F == 16 || F == 32 || F == 64 || F == 128; }
static int launch_k1_h(const float* ref_feature, const uint16_t* vb, const float* homographies, int B, int D, int h, int w,
                       int F, int mode, int out_dtype, uint16_t* o, cudaStream_t st) {
    const int G8 = F / 8;
    const int ppb = 256 / G8, ph = ppb >= 8 ? ppb / 8 : 1, pw = ppb / ph;
    dim3 grid((unsigned)(((w + pw - 1) / pw) * ((h + ph - 1) / ph)), (unsigned)((D + K1_DCHUNK - 1) / K1_DCHUNK), (unsigned)B);
#define K1H(M, G) do { if (out_dtype == ATVS_F16) k_build_cost_volume_h<M, G, true><<<grid, 256, 0, st>>>(ref_feature, vb, homographies, D, h, w, o); \
                       else k_build_cost_volume_h<M, G, false><<<grid, 256, 0, st>>>(ref_feature, vb, homographies, D, h, w, o); } while (0)
#define K1H_G(M) do { switch (G8) { case 1: K1H(M, 1); break; case 2: K1H(M, 2); break; case 4: K1H(M, 4); break; \
                                     case 8: K1H(M, 8); break; default: K1H(M, 16); break; } } while (0)
    if (mode == 0) K1H_G(0);
    else if (mode == 1) K1H_G(1);
    else K1H_G(2);
#undef K1H_G
#undef K1H
    ATVS_LAUNCH_CHECK();
    return 0;
}

extern "C" int atvs_build_cost_volume(const float* ref_feature, const float* view_feature, const float* homographies,
                                      const float* ref_homographies, int B, int D, int h, int w, int F, int mode,
                                      int out_dtype, void* out, atvs_stream_t stream) {
    ATVS_CHECK_ARG(view_feature && homographies && out && (mode == 1 || ref_feature), ATVS_E_NULL,
                   "atvs_build_cost_volume: NULL pointer");
    ATVS_CHECK_ARG(B > 0 && B < 65536 && D > 0 && h > 1 && w > 1 && F > 0, ATVS_E_SHAPE,
                   "atvs_build_cost_volume: bad shape B=%d D=%d h=%d w=%d F=%d", B, D, h, w, F);
    ATVS_CHECK_ARG(mode >= 0 && mode <= 2, ATVS_E_UNSUP, "atvs_build_cost_volume: mode %d", mode);
    ATVS_CHECK_ARG(F % 4 == 0 && (out_dtype == ATVS_F32 || F % 8 == 0), ATVS_E_SHAPE,
                   "atvs_build_cost_volume: F=%d must be a multiple of 4 (8 for 16-bit volumes)", F);
    ATVS_CHECK_ARG((((uintptr_t)ref_feature | (uintptr_t)view_feature | (uintptr_t)out) & 15) == 0, ATVS_E_SHAPE,
                   "atvs_build_cost_volume: buffers must be 16-byte aligned");
    cudaStream_t st = (cudaStream_t)stream;
    if (out_dtype == ATVS_F32)
        return launch_k1<float>(ref_feature, view_feature, homographies, ref_homographies, B, D, h, w, F, mode,
                                (float*)out, st);
    const bool half_out = out_dtype == ATVS_BF16 || out_dtype == ATVS_F16;
    if (half_out && !ref_homographies && k1_h_supported(F)) {
        // 16-bit volume: gather from a 16-bit copy of the source feature map (stream-ordered scratch)
        uint16_t* vb = nullptr;
        const long long n = (long long)B * h * w * F;
        ATVS_CUDA(cudaMallocAsync(&vb, sizeof(uint16_t) * n, st));
        const unsigned cgrid = (unsigned)((n / 4 + 255) / 256 < 2048 ? (n / 4 + 255) / 256 : 2048);
        if (out_dtype == ATVS_F16) k_f32_to_16<true><<<cgrid, 256, 0, st>>>(view_feature, vb, n / 4);
        else k_f32_to_16<false><<<cgrid, 256, 0, st>>>(view_feature, vb, n / 4);
        ATVS_LAUNCH_CHECK();
        const int rc = launch_k1_h(ref_feature, vb, homographies, B, D, h, w, F, mode, out_dtype, (uint16_t*)out, st);
        ATVS_CUDA(cudaFreeAsync(vb, st));
        return rc;
    }
    if (out_dtype == ATVS_BF16)
        return launch_k1<__nv_bfloat16>(ref_feature, view_feature, homographies, ref_homographies, B, D, h, w, F, mode,
                                        (__nv_bfloat16*)out, st);
    if (out_dtype == ATVS_F16)
        return launch_k1<__half>(ref_feature, view_feature, homographies, ref_homographies, B, D, h, w, F, mode,
                                 (__half*)out, st);
    atvs_set_error("atvs_build_cost_volume: out_dtype %d", out_dtype);
    return ATVS_E_DTYPE;
}

extern "C" int atvs_build_cost_volume_src16(const float* ref_feature, const void* view_feature16, const float* homographies,
                                            int B, int D, int h, int w, int F, int mode, int dtype, void* out,
                                            atvs_stream_t stream) {
    ATVS_CHECK_ARG(view_feature16 && homographies && out && (mode == 1 || ref_feature), ATVS_E_NULL,
                   "atvs_build_cost_volume_src16: NULL pointer");
    ATVS_CHECK_ARG(B > 0 && B < 65536 && D > 0 && h > 1 && w > 1, ATVS_E_SHAPE,
                   "atvs_build_cost_volume_src16: bad shape B=%d D=%d h=%d w=%d F=%d", B, D, h, w, F);
    ATVS_CHECK_ARG(mode >= 0 && mode <= 2, ATVS_E_UNSUP, "atvs_build_cost_volume_src16: mode %d", mode);
    ATVS_CHECK_ARG(dtype == ATVS_F16 || dtype == ATVS_BF16, ATVS_E_DTYPE, "atvs_build_cost_volume_src16: dtype %d", dtype);
    ATVS_CHECK_ARG(k1_h_supported(F), ATVS_E_SHAPE, "atvs_build_cost_volume_src16: F=%d (8, 16, 32, 64 or 128)", F);
    ATVS_CHECK_ARG((((uintptr_t)ref_feature | (uintptr_t)view_feature16 | (uintptr_t)out) & 15) == 0, ATVS_E_SHAPE,
                   "atvs_build_cost_volume_src16: buffers must be 16-byte aligned");
    return launch_k1_h(ref_feature, (const uint16_t*)view_feature16, homographies, B, D, h, w, F, mode, dtype, (uint16_t*)out,
                       (cudaStream_t)stream);
}

extern "C" int atvs_prob2depth(const float* prob_volume, int B, int D, int H, int W, const float* depth_start,
                               const float* depth_interval, int up, float* depth, float* prob_map,
                               atvs_stream_t stream) {
    ATVS_CHECK_ARG(prob_volume && depth_start && depth_interval && depth, ATVS_E_NULL, "atvs_prob2depth: NULL pointer");
    ATVS_CHECK_ARG(B > 0 && D > 0 && H > 0 && W > 0, ATVS_E_SHAPE, "atvs_prob2depth: bad shape");
    ATVS_CHECK_ARG(up == 1 || up == 4, ATVS_E_UNSUP, "atvs_prob2depth: up=%d (1 or 4)", up);
    ATVS_CHECK_ARG(up == 1 || (H > 1 && W > 1), ATVS_E_SHAPE, "atvs_prob2depth: up=4 needs H,W > 1");
    const long long total = (long long)B * H * up * W * up;
    const unsigned grid = (unsigned)((total + 255) / 256);
    cudaStream_t st = (cudaStream_t)stream;
    if (up == 1)
    {
        const long long plane = (long long)H * W;
        if (plane % 4 == 0 && total >= 262144 && (((uintptr_t)prob_volume) & 15) == 0)
            k_prob2depth_sliced<4><<<(unsigned)((total + 127) / 128), 256, 0, st>>>(prob_volume, B, D, plane, depth_start,
                                                                                  depth_interval, depth, prob_map);
        else
            k_prob2depth_sliced<1><<<(unsigned)((total + 31) / 32), 256, 0, st>>>(prob_volume, B, D, plane, depth_start,
                                                                                depth_interval, depth, prob_map);
    }
    else
    {
        const int Ho = H * 4;
        const long long blocks = (long long)B * Ho * ((W + 31) / 32);
        if (blocks <= 0x7fffffffLL)
            k_prob2depth_up_sliced<4><<<(unsigned)blocks, 256, 0, st>>>(prob_volume, B, D, H, W, depth_start, depth_interval,
                                                                       depth, prob_map);
        else
            k_prob2depth<4><<<grid, 256, 0, st>>>(prob_volume, B, D, H, W, depth_start, depth_interval, depth, prob_map);
    }
    ATVS_LAUNCH_CHECK();
    return 0;
}
