// net_fp32.cu - CUDA-core fp32 layer primitives of libatvs.so (the fp32 parity path) plus the
// dtype-generic elementwise / batch-norm / attention kernels shared with the bf16 path.
//
//   atvs_conv3d_fp32        <- network.py:142-215 (conv / conv_bn), :511-550 (deconv_bn)
//   atvs_bn_relu_add        <- network.py:206-215, 541-550 (BN with batch statistics, F4) + add :696
//   atvs_attention_*        <- network.py:282-351 (attention_activation), :379-408 (aggregation)
#include "common.cuh"
#include "conv_geom.cuh"

namespace {

// ------------------------------------------------------------------ direct conv, fp32
// one thread = one output voxel x all COUT channels; per-tap weights staged in shared memory;
// grid-stride over 128-voxel tiles so the BN moments are reduced once per CTA.
template <int COUT>
__global__ void __launch_bounds__(128)
k_conv3d_fp32(const float* __restrict__ x, const float* __restrict__ wgt, ConvGeom g, int transposed_w,
              float* __restrict__ out, double* __restrict__ stats, long long njobs) {
    extern __shared__ float ws[];             // [Cin][COUT]
    __shared__ double sstat[2 * COUT];
    const int tid = threadIdx.x;
    const int Cin = g.Cin;
    for (int i = tid; i < 2 * COUT; i += 128) sstat[i] = 0.0;
    const long long ntiles = (njobs + 127) / 128;
    for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const long long j = tile * 128 + tid;
        const bool active = j < njobs;
        long long r = active ? j : 0;
        const int jx = (int)(r % g.Wj); r /= g.Wj;
        const int jy = (int)(r % g.Hj); r /= g.Hj;
        const int jz = (int)(r % g.Dj);
        const int b = (int)(r / g.Dj);
        float acc[COUT];
#pragma unroll
        for (int c = 0; c < COUT; ++c) acc[c] = 0.f;
        for (int tz = 0; tz < g.nt[0]; ++tz)
            for (int ty = 0; ty < g.nt[1]; ++ty)
                for (int tx = 0; tx < g.nt[2]; ++tx) {
                    const int k = (g.kidx[0][tz] * 3 + g.kidx[1][ty]) * 3 + g.kidx[2][tx];
                    __syncthreads();
                    for (int i = tid; i < Cin * COUT; i += 128) {
                        const int ci = i / COUT, co = i % COUT;
                        ws[i] = transposed_w ? __ldg(wgt + ((size_t)k * COUT + co) * Cin + ci)
                                             : __ldg(wgt + ((size_t)k * Cin + ci) * COUT + co);
                    }
                    __syncthreads();
                    const int iz = jz * g.s_in + g.koff[0][tz];
                    const int iy = jy * g.s_in + g.koff[1][ty];
                    const int ix = jx * g.s_in + g.koff[2][tx];
                    const bool ok = active && iz >= 0 && iz < g.Din && iy >= 0 && iy < g.Hin && ix >= 0 && ix < g.Win;
                    if (!ok) continue;
                    const float* xp = x + ((((size_t)b * g.Din + iz) * g.Hin + iy) * g.Win + ix) * Cin;
                    if ((Cin & 3) == 0) {
                        for (int c4 = 0; c4 < Cin; c4 += 4) {
                            const float4 xv = __ldg(reinterpret_cast<const float4*>(xp + c4));
                            const float xs[4] = {xv.x, xv.y, xv.z, xv.w};
#pragma unroll
                            for (int q = 0; q < 4; ++q) {
                                const float* wr = ws + (c4 + q) * COUT;
#pragma unroll
                                for (int c = 0; c < COUT; ++c) acc[c] = fmaf(xs[q], wr[c], acc[c]);
                            }
                        }
                    } else {
                        for (int ci = 0; ci < Cin; ++ci) {
                            const float xv = __ldg(xp + ci);
                            const float* wr = ws + ci * COUT;
#pragma unroll
                            for (int c = 0; c < COUT; ++c) acc[c] = fmaf(xv, wr[c], acc[c]);
                        }
                    }
                }
        if (active) {
            const int oz = jz * g.os + g.p[0], oy = jy * g.os + g.p[1], ox = jx * g.os + g.p[2];
            float* op = out + ((((size_t)b * g.Do + oz) * g.Ho + oy) * g.Wo + ox) * COUT;
            if (COUT % 4 == 0) {
#pragma unroll
                for (int c = 0; c < COUT; c += 4)
                    *reinterpret_cast<float4*>(op + c) = make_float4(acc[c], acc[c + 1], acc[c + 2], acc[c + 3]);
            } else {
#pragma unroll
                for (int c = 0; c < COUT; ++c) op[c] = acc[c];
            }
        }
        if (stats) {
#pragma unroll
            for (int c = 0; c < COUT; ++c) {
                float s = active ? acc[c] : 0.f;
                float q = s * s;
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
                    s += __shfl_xor_sync(0xffffffffu, s, o);
                    q += __shfl_xor_sync(0xffffffffu, q, o);
                }
                if ((tid & 31) == 0) {
                    atomicAdd(&sstat[c], (double)s);
                    atomicAdd(&sstat[COUT + c], (double)q);
                }
            }
        }
    }
    if (stats) {
        __syncthreads();
        for (int i = tid; i < 2 * COUT; i += 128) atomicAdd(&stats[i], sstat[i]);
    }
}

// ------------------------------------------------------------------ BN + ReLU + adds
template <typename T>
struct Vec4 {};
template <>
struct Vec4<float> {
    static __device__ __forceinline__ float4 ld(const float* p) { return *reinterpret_cast<const float4*>(p); }
    static __device__ __forceinline__ void st(float* p, float4 v) { *reinterpret_cast<float4*>(p) = v; }
    static __device__ __forceinline__ float ld1(const float* p) { return *p; }
    static __device__ __forceinline__ void st1(float* p, float v) { *p = v; }
};
template <>
struct Vec4<__nv_bfloat16> {
    static __device__ __forceinline__ float4 ld(const __nv_bfloat16* p) {
        const uint2 u = *reinterpret_cast<const uint2*>(p);
        const __nv_bfloat162 a = *reinterpret_cast<const __nv_bfloat162*>(&u.x);
        const __nv_bfloat162 b = *reinterpret_cast<const __nv_bfloat162*>(&u.y);
        const float2 fa = __bfloat1622float2(a), fb = __bfloat1622float2(b);
        return make_float4(fa.x, fa.y, fb.x, fb.y);
    }
    static __device__ __forceinline__ void st(__nv_bfloat16* p, float4 v) {
        __nv_bfloat162 lo = __floats2bfloat162_rn(v.x, v.y), hi = __floats2bfloat162_rn(v.z, v.w);
        uint2 u;
        u.x = *reinterpret_cast<unsigned*>(&lo);
        u.y = *reinterpret_cast<unsigned*>(&hi);
        *reinterpret_cast<uint2*>(p) = u;
    }
    static __device__ __forceinline__ float ld1(const __nv_bfloat16* p) { return __bfloat162float(*p); }
    static __device__ __forceinline__ void st1(__nv_bfloat16* p, float v) { *p = __float2bfloat16_rn(v); }
};

__device__ __forceinline__ unsigned h2_sat(float lo, float hi) {
    unsigned r;
    asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
    return r;
}
__device__ __forceinline__ float2 h2_f2(unsigned u) { return __half22float2(*reinterpret_cast<const __half2*>(&u)); }
template <>
struct Vec4<__half> {
    static __device__ __forceinline__ float4 ld(const __half* p) {
        const uint2 u = *reinterpret_cast<const uint2*>(p);
        const float2 a = h2_f2(u.x), b = h2_f2(u.y);
        return make_float4(a.x, a.y, b.x, b.y);
    }
    static __device__ __forceinline__ void st(__half* p, float4 v) {
        uint2 u;
        u.x = h2_sat(v.x, v.y);
        u.y = h2_sat(v.z, v.w);
        *reinterpret_cast<uint2*>(p) = u;
    }
    static __device__ __forceinline__ float ld1(const __half* p) { return __half2float(*p); }
    static __device__ __forceinline__ void st1(__half* p, float v) {
        *reinterpret_cast<unsigned short*>(p) = (unsigned short)(h2_sat(v, 0.f) & 0xffffu);
    }
};

template <typename T>
struct Vec8 {};
template <>
struct Vec8<__half> {
    static __device__ __forceinline__ void ld(const __half* p, float4& a, float4& b) {
        const uint4 u = *reinterpret_cast<const uint4*>(p);
        const float2 x = h2_f2(u.x), y = h2_f2(u.y), z = h2_f2(u.z), w = h2_f2(u.w);
        a = make_float4(x.x, x.y, y.x, y.y);
        b = make_float4(z.x, z.y, w.x, w.y);
    }
    static __device__ __forceinline__ void st(__half* p, float4 a, float4 b) {
        uint4 u;
        u.x = h2_sat(a.x, a.y); u.y = h2_sat(a.z, a.w); u.z = h2_sat(b.x, b.y); u.w = h2_sat(b.z, b.w);
        *reinterpret_cast<uint4*>(p) = u;
    }
};
template <>
struct Vec8<float> {
    static __device__ __forceinline__ void ld(const float* p, float4& a, float4& b) {
        a = *reinterpret_cast<const float4*>(p);
        b = *(reinterpret_cast<const float4*>(p) + 1);
    }
    static __device__ __forceinline__ void st(float* p, float4 a, float4 b) {
        *reinterpret_cast<float4*>(p) = a;
        *(reinterpret_cast<float4*>(p) + 1) = b;
    }
};
template <>
struct Vec8<__nv_bfloat16> {
    static __device__ __forceinline__ void ld(const __nv_bfloat16* p, float4& a, float4& b) {
        const uint4 u = *reinterpret_cast<const uint4*>(p);
        const float2 f0 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u.x));
        const float2 f1 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u.y));
        const float2 f2 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u.z));
        const float2 f3 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u.w));
        a = make_float4(f0.x, f0.y, f1.x, f1.y);
        b = make_float4(f2.x, f2.y, f3.x, f3.y);
    }
    static __device__ __forceinline__ void st(__nv_bfloat16* p, float4 a, float4 b) {
        __nv_bfloat162 q0 = __floats2bfloat162_rn(a.x, a.y), q1 = __floats2bfloat162_rn(a.z, a.w);
        __nv_bfloat162 q2 = __floats2bfloat162_rn(b.x, b.y), q3 = __floats2bfloat162_rn(b.z, b.w);
        uint4 u;
        u.x = *reinterpret_cast<unsigned*>(&q0); u.y = *reinterpret_cast<unsigned*>(&q1);
        u.z = *reinterpret_cast<unsigned*>(&q2); u.w = *reinterpret_cast<unsigned*>(&q3);
        *reinterpret_cast<uint4*>(p) = u;
    }
};

constexpr int BN_MAXC = 256;

// out = relu((raw - mean) * rsqrt(var + eps))  [+ relu(bn(raw2))] [+ s1] [+ s2]
//   batch statistics from the fp64 moment sums (network.py:206-212, training=True, no affine).
//   raw2/stats2: a SECOND raw convolution output joined by the same `add` (network.py:696), so that
//   a layer whose only consumer is that add never has its normalised tensor written and re-read.
// 8 elements per thread and iteration when C is a multiple of 8: two 16-byte raw loads, one 16-byte
// bf16 store.
// raw tensors are fp32 or fp16 (RawT): 8 / 4 / 1 consecutive values as fp32
template <typename RawT> struct RawLd;
template <> struct RawLd<float> {
    static __device__ __forceinline__ void ld8(const float* p, float4& a, float4& b) {
        // one 32-byte load when the row is 32-byte aligned is not guaranteed here (16-byte contract): two LDG.128
        a = __ldcs(reinterpret_cast<const float4*>(p)); b = __ldcs(reinterpret_cast<const float4*>(p) + 1);
    }
    static __device__ __forceinline__ float4 ld4(const float* p) { return __ldcs(reinterpret_cast<const float4*>(p)); }
    static __device__ __forceinline__ float ld1(const float* p) { return *p; }
};
template <> struct RawLd<__half> {
    static __device__ __forceinline__ float2 h2(unsigned u) { return __half22float2(*reinterpret_cast<const __half2*>(&u)); }
    static __device__ __forceinline__ void ld8(const __half* p, float4& a, float4& b) {
        const uint4 u = __ldcs(reinterpret_cast<const uint4*>(p));
        const float2 x = h2(u.x), y = h2(u.y), z = h2(u.z), w = h2(u.w);
        a = make_float4(x.x, x.y, y.x, y.y); b = make_float4(z.x, z.y, w.x, w.y);
    }
    static __device__ __forceinline__ float4 ld4(const __half* p) {
        const uint2 u = __ldcs(reinterpret_cast<const uint2*>(p));
        const float2 x = h2(u.x), y = h2(u.y);
        return make_float4(x.x, x.y, y.x, y.y);
    }
    static __device__ __forceinline__ float ld1(const __half* p) { return __half2float(*p); }
};

// 8 consecutive elements as they sit in memory (16 bytes for bf16 / fp16, 32 for fp32): loads are issued in this form
// and unpacked to fp32 only when used, so that several of them can be in flight per thread at 16 registers
template <typename E> struct Pk8 { uint4 u; };
template <> struct Pk8<float> { float4 a, b; };
template <typename E>
__device__ __forceinline__ Pk8<E> ldp8(const E* p) {
    Pk8<E> r;
    r.u = __ldcs(reinterpret_cast<const uint4*>(p));
    return r;
}
template <>
__device__ __forceinline__ Pk8<float> ldp8<float>(const float* p) {
    Pk8<float> r;
    r.a = __ldcs(reinterpret_cast<const float4*>(p));
    r.b = __ldcs(reinterpret_cast<const float4*>(p) + 1);
    return r;
}
__device__ __forceinline__ void unpack8(const Pk8<float>& k, float4& a, float4& b) { a = k.a; b = k.b; }
__device__ __forceinline__ void unpack8(const Pk8<__half>& k, float4& a, float4& b) {
    const float2 x = RawLd<__half>::h2(k.u.x), y = RawLd<__half>::h2(k.u.y), z = RawLd<__half>::h2(k.u.z), w = RawLd<__half>::h2(k.u.w);
    a = make_float4(x.x, x.y, y.x, y.y); b = make_float4(z.x, z.y, w.x, w.y);
}
__device__ __forceinline__ void unpack8(const Pk8<__nv_bfloat16>& k, float4& a, float4& b) {
    a = make_float4(__uint_as_float(k.u.x << 16), __uint_as_float(k.u.x & 0xffff0000u), __uint_as_float(k.u.y << 16),
                    __uint_as_float(k.u.y & 0xffff0000u));
    b = make_float4(__uint_as_float(k.u.z << 16), __uint_as_float(k.u.z & 0xffff0000u), __uint_as_float(k.u.w << 16),
                    __uint_as_float(k.u.w & 0xffff0000u));
}

template <typename T, typename RawT>
__global__ void __launch_bounds__(256)
k_bn_relu_add(const RawT* __restrict__ raw, const double* __restrict__ stats, const RawT* __restrict__ raw2,
              const double* __restrict__ stats2, long long count, int C, float eps, int relu,
              const T* __restrict__ s1, const T* __restrict__ s2, T* __restrict__ out_plain, T* __restrict__ out_sum) {
    __shared__ float sh_inv[BN_MAXC], sh_off[BN_MAXC], sh_inv2[BN_MAXC], sh_off2[BN_MAXC];
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
        float inv = 1.f, off = 0.f, inv2 = 1.f, off2 = 0.f;
        if (stats) {
            const double mean = stats[c] / (double)count;
            double var = stats[C + c] / (double)count - mean * mean;
            if (var < 0.0) var = 0.0;
            inv = (float)(1.0 / sqrt(var + (double)eps));
            off = (float)mean * inv;
        }
        if (stats2) {
            const double mean = stats2[c] / (double)count;
            double var = stats2[C + c] / (double)count - mean * mean;
            if (var < 0.0) var = 0.0;
            inv2 = (float)(1.0 / sqrt(var + (double)eps));
            off2 = (float)mean * inv2;
        }
        sh_inv[c] = inv; sh_off[c] = off; sh_inv2[c] = inv2; sh_off2[c] = off2;
    }
    __syncthreads();
    const long long n = count * C;
    auto norm4 = [&](float4 r, const float* inv, const float* off, int c) {
        float4 y;
        y.x = r.x * inv[c] - off[c];
        y.y = r.y * inv[c + 1] - off[c + 1];
        y.z = r.z * inv[c + 2] - off[c + 2];
        y.w = r.w * inv[c + 3] - off[c + 3];
        if (relu) { y.x = fmaxf(y.x, 0.f); y.y = fmaxf(y.y, 0.f); y.z = fmaxf(y.z, 0.f); y.w = fmaxf(y.w, 0.f); }
        return y;
    };
    auto add4 = [](float4& y, float4 a) { y.x += a.x; y.y += a.y; y.z += a.z; y.w += a.w; };
    if ((C & 7) == 0) {
        const long long n8 = n >> 3;
        const bool pow2 = (C & (C - 1)) == 0;
        // two 8-element groups per thread and iteration, every load of both issued before the first use: with ~1500
        // resident threads per SM one 16-byte load each is not enough bytes in flight to cover the HBM latency
        constexpr int U = 2;
        const long long stride = (long long)gridDim.x * blockDim.x;
        const bool sum_in = out_sum != nullptr;
        for (long long i0 = (long long)blockIdx.x * blockDim.x + threadIdx.x; i0 < n8; i0 += U * stride) {
            long long e[U];
            bool ok[U];
            Pk8<RawT> pr[U], pq[U];
            Pk8<T> p1[U], p2[U];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const long long i = i0 + u * stride;
                ok[u] = i < n8;
                e[u] = (ok[u] ? i : i0) << 3;
            }
#pragma unroll
            for (int u = 0; u < U; ++u) {
                pr[u] = ldp8<RawT>(raw + e[u]);
                if (sum_in && raw2) pq[u] = ldp8<RawT>(raw2 + e[u]);
                if (sum_in && s1) p1[u] = ldp8<T>(s1 + e[u]);
                if (sum_in && s2) p2[u] = ldp8<T>(s2 + e[u]);
            }
#pragma unroll
            for (int u = 0; u < U; ++u) {
                if (!ok[u]) continue;
                const int c = pow2 ? (int)(e[u] & (C - 1)) : (int)(e[u] % C);
                float4 ta, tb;
                unpack8(pr[u], ta, tb);
                float4 ya = norm4(ta, sh_inv, sh_off, c);
                float4 yb = norm4(tb, sh_inv, sh_off, c + 4);
                if (out_plain) Vec8<T>::st(out_plain + e[u], ya, yb);
                if (sum_in) {
                    if (raw2) {
                        unpack8(pq[u], ta, tb);
                        add4(ya, norm4(ta, sh_inv2, sh_off2, c));
                        add4(yb, norm4(tb, sh_inv2, sh_off2, c + 4));
                    }
                    if (s1) { unpack8(p1[u], ta, tb); add4(ya, ta); add4(yb, tb); }
                    if (s2) { unpack8(p2[u], ta, tb); add4(ya, ta); add4(yb, tb); }
                    Vec8<T>::st(out_sum + e[u], ya, yb);
                }
            }
        }
    } else if ((C & 3) == 0) {
        const long long n4 = n >> 2;
        for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4;
             i += (long long)gridDim.x * blockDim.x) {
            const int c = (int)((i << 2) % C);
            float4 y = norm4(RawLd<RawT>::ld4(raw + (i << 2)), sh_inv, sh_off, c);
            if (out_plain) Vec4<T>::st(out_plain + (i << 2), y);
            if (out_sum) {
                if (raw2) add4(y, norm4(RawLd<RawT>::ld4(raw2 + (i << 2)), sh_inv2, sh_off2, c));
                if (s1) add4(y, Vec4<T>::ld(s1 + (i << 2)));
                if (s2) add4(y, Vec4<T>::ld(s2 + (i << 2)));
                Vec4<T>::st(out_sum + (i << 2), y);
            }
        }
    } else {
        for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n;
             i += (long long)gridDim.x * blockDim.x) {
            const int c = (int)(i % C);
            float y = RawLd<RawT>::ld1(raw + i) * sh_inv[c] - sh_off[c];
            if (relu) y = fmaxf(y, 0.f);
            if (out_plain) Vec4<T>::st1(out_plain + i, y);
            if (out_sum) {
                if (raw2) {
                    float y2 = RawLd<RawT>::ld1(raw2 + i) * sh_inv2[c] - sh_off2[c];
                    if (relu) y2 = fmaxf(y2, 0.f);
                    y += y2;
                }
                if (s1) y += Vec4<T>::ld1(s1 + i);
                if (s2) y += Vec4<T>::ld1(s2 + i);
                Vec4<T>::st1(out_sum + i, y);
            }
        }
    }
}

template <typename TS, typename TD>
__global__ void k_cast(const TS* __restrict__ s, TD* __restrict__ d, long long n) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
        Vec4<TD>::st1(d + i, Vec4<TS>::ld1(s + i));
}

template <typename T>
__global__ void k_add(const T* __restrict__ a, const T* __restrict__ b, T* __restrict__ o, long long n) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
        Vec4<T>::st1(o + i, Vec4<T>::ld1(a + i) + Vec4<T>::ld1(b + i));
}

// ------------------------------------------------------------------ attention (AAM)
constexpr int ATT_MAXN = 8;

// MODE 0: full softmax-weighted sum (single GPU, reference order incl. the +S term)
// MODE 1: local max of l_n = u_n - s_n
// MODE 2: partial numerator || denominator against a given max
template <typename T, int MODE>
__global__ void __launch_bounds__(256)
k_attention(const T* __restrict__ act, const T* __restrict__ x, int N, long long V, int C, const float* __restrict__ gmax,
            float* __restrict__ out) {
    const int G = C >> 2;
    const long long total = V * G;
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
         idx += (long long)gridDim.x * blockDim.x) {
        const long long v = idx / G;
        const int c0 = (int)(idx % G) << 2;
        float4 u[ATT_MAXN], s[ATT_MAXN];
#pragma unroll
        for (int n = 0; n < ATT_MAXN; ++n) {
            if (n < N) {
                const T* a = act + ((size_t)n * V + v) * (2 * C);
                u[n] = Vec4<T>::ld(a + c0);
                s[n] = Vec4<T>::ld(a + C + c0);
            }
        }
        float res[4], den[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            float S = 0.f;
            if (MODE == 0) {
#pragma unroll
                for (int n = 0; n < ATT_MAXN; ++n)
                    if (n < N) S = (n == 0) ? (&s[n].x)[q] : S + (&s[n].x)[q];
            }
            float a[ATT_MAXN];
            float m = -INFINITY;
#pragma unroll
            for (int n = 0; n < ATT_MAXN; ++n)
                if (n < N) {
                    a[n] = ((&u[n].x)[q] - (&s[n].x)[q]) + S;
                    m = fmaxf(m, a[n]);
                }
            if (MODE == 1) { res[q] = m; continue; }
            if (MODE == 2) m = gmax[v * C + c0 + q];
            float dsum = 0.f;
#pragma unroll
            for (int n = 0; n < ATT_MAXN; ++n)
                if (n < N) {
                    a[n] = expf(a[n] - m);
                    dsum += a[n];
                }
            float r = 0.f;
#pragma unroll
            for (int n = 0; n < ATT_MAXN; ++n)
                if (n < N) {
                    const float xv = Vec4<T>::ld1(x + ((size_t)n * V + v) * C + c0 + q);
                    r += (MODE == 0 ? a[n] / dsum : a[n]) * xv;
                }
            res[q] = r;
            den[q] = dsum;
        }
        if (MODE == 2) {
            *reinterpret_cast<float4*>(out + v * (2 * C) + c0) = make_float4(res[0], res[1], res[2], res[3]);
            *reinterpret_cast<float4*>(out + v * (2 * C) + C + c0) = make_float4(den[0], den[1], den[2], den[3]);
        } else {
            *reinterpret_cast<float4*>(out + v * C + c0) = make_float4(res[0], res[1], res[2], res[3]);
        }
    }
}


// AAM on the RAW attention convolutions: act_raw (N,V,2C) fp32 is the un-activated output of the one
// 8->16 convolution per view ([W_unique | W_shared], network.py:313-344); the ReLU is applied while
// loading, so the activations are never written back and re-read, and one thread owns 8 channels of a
// voxel (16/32-byte loads).  Same three modes as k_attention.
// the N per-view cost volumes (V,C) by pointer: the views stay where stage I wrote them (no stacking copy)
struct AttViews {
    const void* p[ATT_MAXN];
};

template <typename T, typename ActT, int MODE, int NMAX>
__global__ void __launch_bounds__(256)
k_attention_raw(const ActT* __restrict__ act, const AttViews xs, int N, long long V, int C,
                const float* __restrict__ gmax, float* __restrict__ out) {
    const int G = C >> 3;
    const long long total = V * G;
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
         idx += (long long)gridDim.x * blockDim.x) {
        const long long v = idx / G;
        const int c0 = (int)(idx % G) << 3;
        float a[NMAX][8];
        float S[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) S[q] = 0.f;
#pragma unroll
        for (int n = 0; n < NMAX; ++n) {
            if (n < N) {
                const ActT* ar = act + ((size_t)n * V + v) * (2 * C);
                float4 u0, u1, s0, s1;
                RawLd<ActT>::ld8(ar + c0, u0, u1);
                RawLd<ActT>::ld8(ar + C + c0, s0, s1);
                const float uu[8] = {u0.x, u0.y, u0.z, u0.w, u1.x, u1.y, u1.z, u1.w};
                const float ss[8] = {s0.x, s0.y, s0.z, s0.w, s1.x, s1.y, s1.z, s1.w};
#pragma unroll
                for (int q = 0; q < 8; ++q) {
                    const float sq = fmaxf(ss[q], 0.f);
                    a[n][q] = fmaxf(uu[q], 0.f) - sq;
                    if (MODE == 0) S[q] = (n == 0) ? sq : S[q] + sq;
                }
            }
        }
        float m[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            float mm = -INFINITY;
#pragma unroll
            for (int n = 0; n < NMAX; ++n)
                if (n < N) {
                    a[n][q] += S[q];
                    mm = fmaxf(mm, a[n][q]);
                }
            m[q] = mm;
        }
        if (MODE == 1) {
            Vec8<float>::st(out + v * C + c0, make_float4(m[0], m[1], m[2], m[3]), make_float4(m[4], m[5], m[6], m[7]));
            continue;
        }
        if (MODE == 2) {
            float4 g0, g1;
            Vec8<float>::ld(gmax + v * C + c0, g0, g1);
            m[0] = g0.x; m[1] = g0.y; m[2] = g0.z; m[3] = g0.w; m[4] = g1.x; m[5] = g1.y; m[6] = g1.z; m[7] = g1.w;
        }
        float den[8], res[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) { den[q] = 0.f; res[q] = 0.f; }
#pragma unroll
        for (int n = 0; n < NMAX; ++n)
            if (n < N) {
#pragma unroll
                for (int q = 0; q < 8; ++q) {
                    // bf16 activations: SFU exponential (the weights are rounded to 8 bits downstream anyway)
                    a[n][q] = (sizeof(T) == 4) ? expf(a[n][q] - m[q]) : exp2f((a[n][q] - m[q]) * 1.4426950408889634f);
                    den[q] += a[n][q];
                }
            }
        float inv[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) inv[q] = 1.0f / den[q];
#pragma unroll
        for (int n = 0; n < NMAX; ++n)
            if (n < N) {
                float4 x0, x1;
                Vec8<T>::ld(reinterpret_cast<const T*>(xs.p[n]) + (size_t)v * C + c0, x0, x1);
                const float xx[8] = {x0.x, x0.y, x0.z, x0.w, x1.x, x1.y, x1.z, x1.w};
#pragma unroll
                for (int q = 0; q < 8; ++q) {
                    // fp32 path: the reference's e / sum, then * x (network.py:402-406); bf16 path: one reciprocal per channel
                    const float sc = (MODE != 0) ? a[n][q] : ((sizeof(T) == 4) ? a[n][q] / den[q] : a[n][q] * inv[q]);
                    res[q] += sc * xx[q];
                }
            }
        if (MODE == 2) {
            Vec8<float>::st(out + v * (2 * C) + c0, make_float4(res[0], res[1], res[2], res[3]),
                            make_float4(res[4], res[5], res[6], res[7]));
            Vec8<float>::st(out + v * (2 * C) + C + c0, make_float4(den[0], den[1], den[2], den[3]),
                            make_float4(den[4], den[5], den[6], den[7]));
        } else {
            Vec8<float>::st(out + v * C + c0, make_float4(res[0], res[1], res[2], res[3]),
                            make_float4(res[4], res[5], res[6], res[7]));
        }
    }
}

__global__ void k_attention_finish(const float* __restrict__ nd, long long V, int C, float* __restrict__ out) {
    const long long total = V * C;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
         i += (long long)gridDim.x * blockDim.x) {
        const long long v = i / C;
        const int c = (int)(i % C);
        out[i] = nd[v * 2 * C + c] / nd[v * 2 * C + C + c];
    }
}

inline unsigned grid_for(long long n, int block, int per_sm) {
    long long g = (n + block - 1) / block;
    const long long cap = (long long)atvs_num_sms() * per_sm;
    if (g > cap) g = cap;
    if (g < 1) g = 1;
    return (unsigned)g;
}

}  // namespace

// =========================================================================== C ABI
extern "C" int atvs_conv3d_fp32(const float* x, const float* kernel, int B, int D, int H, int W, int Cin, int Cout,
                                int stride, int transposed, float* raw_out, double* stats, atvs_stream_t stream) {
    ATVS_CHECK_ARG(x && kernel && raw_out, ATVS_E_NULL, "atvs_conv3d_fp32: NULL pointer");
    ATVS_CHECK_ARG(B > 0 && D > 0 && H > 0 && W > 0 && Cin > 0 && Cin <= 256, ATVS_E_SHAPE,
                   "atvs_conv3d_fp32: bad shape");
    ATVS_CHECK_ARG(transposed ? stride == 2 : (stride == 1 || stride == 2), ATVS_E_UNSUP,
                   "atvs_conv3d_fp32: stride=%d transposed=%d", stride, transposed);
    ATVS_CHECK_ARG(Cout == 1 || Cout == 8 || Cout == 16 || Cout == 32 || Cout == 64, ATVS_E_UNSUP,
                   "atvs_conv3d_fp32: Cout=%d (1, 8, 16, 32 or 64)", Cout);
    cudaStream_t st = (cudaStream_t)stream;
    const int ncls = transposed ? 8 : 1;
    for (int cls = 0; cls < ncls; ++cls) {
        const ConvGeom g = make_conv_geom(B, D, H, W, Cin, Cout, stride, transposed, cls);
        const long long njobs = (long long)B * g.Dj * g.Hj * g.Wj;
        const unsigned grid = grid_for(njobs, 128, 8);
        const size_t smem = sizeof(float) * (size_t)Cin * Cout;
#define CONV_GO(CO)                                                                                              \
    k_conv3d_fp32<CO><<<grid, 128, smem, st>>>(x, kernel, g, transposed, raw_out, stats, njobs)
        switch (Cout) {
            case 1: CONV_GO(1); break;
            case 8: CONV_GO(8); break;
            case 16: CONV_GO(16); break;
            case 32: CONV_GO(32); break;
            default: CONV_GO(64); break;
        }
#undef CONV_GO
        ATVS_LAUNCH_CHECK();
    }
    return 0;
}

// grid of a grid-stride kernel = exactly the blocks that are resident at once (occupancy API, cached per kernel and
// device): a grid of 8 blocks per SM with 6 resident runs as 1.33 waves and idles a third of the machine in the second one
template <auto KERNEL>
static unsigned grid_resident(long long n, int block) {
    static std::atomic<int> per_sm[ATVS_MAX_DEVICES];       // 0 = not queried yet on that device
    int dev = 0;
    if (atvs_current_device(&dev) != 0) return grid_for(n, block, 4);
    int b = per_sm[dev].load(std::memory_order_relaxed);
    if (b == 0) {
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&b, KERNEL, block, 0) != cudaSuccess || b < 1) b = 4;
        per_sm[dev].store(b, std::memory_order_relaxed);
    }
    return grid_for(n, block, b);
}

template <typename RawT>
static int bn_relu_add_launch(const RawT* raw, const double* stats, const RawT* raw2, const double* stats2, long long count,
                              int C, float eps, int relu, const void* skip1, const void* skip2, void* out_plain,
                              void* out_sum, int act_dtype, cudaStream_t st, const char* who) {
    if (act_dtype == ATVS_F32) {
        const unsigned grid = grid_resident<k_bn_relu_add<float, RawT>>(count * C / 8 + 1, 256);
        k_bn_relu_add<float, RawT><<<grid, 256, 0, st>>>(raw, stats, raw2, stats2, count, C, eps, relu, (const float*)skip1,
                                                         (const float*)skip2, (float*)out_plain, (float*)out_sum);
    } else if (act_dtype == ATVS_BF16) {
        const unsigned grid = grid_resident<k_bn_relu_add<__nv_bfloat16, RawT>>(count * C / 8 + 1, 256);
        k_bn_relu_add<__nv_bfloat16, RawT><<<grid, 256, 0, st>>>(raw, stats, raw2, stats2, count, C, eps, relu,
                                                                 (const __nv_bfloat16*)skip1, (const __nv_bfloat16*)skip2,
                                                                 (__nv_bfloat16*)out_plain, (__nv_bfloat16*)out_sum);
    } else if (act_dtype == ATVS_F16) {
        const unsigned grid = grid_resident<k_bn_relu_add<__half, RawT>>(count * C / 8 + 1, 256);
        k_bn_relu_add<__half, RawT><<<grid, 256, 0, st>>>(raw, stats, raw2, stats2, count, C, eps, relu, (const __half*)skip1,
                                                          (const __half*)skip2, (__half*)out_plain, (__half*)out_sum);
    } else {
        atvs_set_error("%s: act_dtype %d", who, act_dtype);
        return ATVS_E_DTYPE;
    }
    ATVS_LAUNCH_CHECK();
    return 0;
}

static int bn_relu_add_impl(const void* raw, const double* stats, const void* raw2, const double* stats2, int raw_dtype,
                            long long count, int C, float eps, int relu, const void* skip1, const void* skip2,
                            void* out_plain, void* out_sum, int act_dtype, cudaStream_t st, const char* who) {
    ATVS_CHECK_ARG(raw && (out_plain || out_sum), ATVS_E_NULL, "%s: NULL pointer", who);
    ATVS_CHECK_ARG(count > 0 && C > 0 && C <= BN_MAXC, ATVS_E_SHAPE, "%s: count=%lld C=%d", who, count, C);
    ATVS_CHECK_ARG(raw_dtype == ATVS_F32 || raw_dtype == ATVS_F16, ATVS_E_DTYPE, "%s: raw_dtype %d", who, raw_dtype);
    ATVS_CHECK_ARG((C & 3) != 0 || (((uintptr_t)raw | (uintptr_t)raw2 | (uintptr_t)skip1 | (uintptr_t)skip2 |
                                      (uintptr_t)out_plain | (uintptr_t)out_sum) & 15) == 0,
                   ATVS_E_SHAPE, "%s: buffers must be 16-byte aligned", who);
    if (raw_dtype == ATVS_F16)
        return bn_relu_add_launch<__half>((const __half*)raw, stats, (const __half*)raw2, stats2, count, C, eps, relu, skip1,
                                          skip2, out_plain, out_sum, act_dtype, st, who);
    return bn_relu_add_launch<float>((const float*)raw, stats, (const float*)raw2, stats2, count, C, eps, relu, skip1, skip2,
                                     out_plain, out_sum, act_dtype, st, who);
}

extern "C" int atvs_bn_relu_add(const void* raw, int raw_dtype, const double* stats, long long count, int C, float eps,
                                int relu, const void* skip1, const void* skip2, void* out_plain, void* out_sum,
                                int act_dtype, atvs_stream_t stream) {
    return bn_relu_add_impl(raw, stats, nullptr, nullptr, raw_dtype, count, C, eps, relu, skip1, skip2, out_plain, out_sum,
                            act_dtype, (cudaStream_t)stream, "atvs_bn_relu_add");
}

extern "C" int atvs_bn_relu_add_pair(const void* raw_a, const double* stats_a, const void* raw_b, const double* stats_b,
                                     int raw_dtype, long long count, int C, float eps, int relu, const void* skip,
                                     void* out_plain_a, void* out_sum, int act_dtype, atvs_stream_t stream) {
    ATVS_CHECK_ARG(raw_b && out_sum, ATVS_E_NULL, "atvs_bn_relu_add_pair: NULL pointer");
    return bn_relu_add_impl(raw_a, stats_a, raw_b, stats_b, raw_dtype, count, C, eps, relu, skip, nullptr, out_plain_a,
                            out_sum, act_dtype, (cudaStream_t)stream, "atvs_bn_relu_add_pair");
}

extern "C" int atvs_cast(const void* src, int src_dtype, void* dst, int dst_dtype, long long n, atvs_stream_t stream) {
    ATVS_CHECK_ARG(src && dst, ATVS_E_NULL, "atvs_cast: NULL pointer");
    ATVS_CHECK_ARG(n >= 0, ATVS_E_SHAPE, "atvs_cast: n=%lld", n);
    if (n == 0) return 0;
    cudaStream_t st = (cudaStream_t)stream;
    const unsigned grid = grid_for(n, 256, 8);
    if (src_dtype == ATVS_F32 && dst_dtype == ATVS_BF16)
        k_cast<float, __nv_bfloat16><<<grid, 256, 0, st>>>((const float*)src, (__nv_bfloat16*)dst, n);
    else if (src_dtype == ATVS_BF16 && dst_dtype == ATVS_F32)
        k_cast<__nv_bfloat16, float><<<grid, 256, 0, st>>>((const __nv_bfloat16*)src, (float*)dst, n);
    else if (src_dtype == ATVS_F32 && dst_dtype == ATVS_F32)
        k_cast<float, float><<<grid, 256, 0, st>>>((const float*)src, (float*)dst, n);
    else if (src_dtype == ATVS_BF16 && dst_dtype == ATVS_BF16)
        k_cast<__nv_bfloat16, __nv_bfloat16><<<grid, 256, 0, st>>>((const __nv_bfloat16*)src, (__nv_bfloat16*)dst, n);
    else if (src_dtype == ATVS_F32 && dst_dtype == ATVS_F16)
        k_cast<float, __half><<<grid, 256, 0, st>>>((const float*)src, (__half*)dst, n);
    else if (src_dtype == ATVS_F16 && dst_dtype == ATVS_F32)
        k_cast<__half, float><<<grid, 256, 0, st>>>((const __half*)src, (float*)dst, n);
    else if (src_dtype == ATVS_F16 && dst_dtype == ATVS_F16)
        k_cast<__half, __half><<<grid, 256, 0, st>>>((const __half*)src, (__half*)dst, n);
    else {
        atvs_set_error("atvs_cast: dtype %d -> %d", src_dtype, dst_dtype);
        return ATVS_E_DTYPE;
    }
    ATVS_LAUNCH_CHECK();
    return 0;
}

// fp32 rows of C channels -> 16-bit rows of Cpad >= C channels, the extra channels zero: one pass instead of
// zero fill + strided copy + cast (the refinement U-Net's 48 / 19 / 1-channel input groups, refine._pad_channels)
template <typename OutT>
__global__ void __launch_bounds__(256)
k_pad_cast(const float* __restrict__ x, long long rows, int C, int Cpad, OutT* __restrict__ out) {
    const long long n = rows * (long long)(Cpad >> 3);          // one thread per 8 output channels (16 bytes)
    const int g8 = Cpad >> 3;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const long long r = i / g8;
        const int c0 = (int)(i - r * g8) << 3;
        const float* src = x + r * C + c0;
        OutT v[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) v[k] = (OutT)((c0 + k < C) ? __ldg(src + k) : 0.f);
        *reinterpret_cast<uint4*>(out + r * Cpad + c0) = *reinterpret_cast<const uint4*>(v);
    }
}

extern "C" int atvs_pad_cast(const float* x, long long rows, int C, int Cpad, void* out, int out_dtype, atvs_stream_t stream) {
    ATVS_CHECK_ARG(x && out, ATVS_E_NULL, "atvs_pad_cast: NULL pointer");
    ATVS_CHECK_ARG(rows > 0 && C > 0 && Cpad >= C && (Cpad & 7) == 0, ATVS_E_SHAPE, "atvs_pad_cast: rows=%lld C=%d Cpad=%d (Cpad >= C, multiple of 8)", rows, C, Cpad);
    ATVS_CHECK_ARG(((uintptr_t)out & 15) == 0, ATVS_E_SHAPE, "atvs_pad_cast: out must be 16-byte aligned");
    const unsigned grid = grid_for(rows * (Cpad >> 3), 256, 4);
    if (out_dtype == ATVS_F16) k_pad_cast<__half><<<grid, 256, 0, (cudaStream_t)stream>>>(x, rows, C, Cpad, (__half*)out);
    else if (out_dtype == ATVS_BF16) k_pad_cast<__nv_bfloat16><<<grid, 256, 0, (cudaStream_t)stream>>>(x, rows, C, Cpad, (__nv_bfloat16*)out);
    else {
        atvs_set_error("atvs_pad_cast: out_dtype %d (ATVS_F16 | ATVS_BF16)", out_dtype);
        return ATVS_E_DTYPE;
    }
    ATVS_LAUNCH_CHECK();
    return 0;
}

extern "C" int atvs_add(const void* a, const void* b, void* out, int dtype, long long n, atvs_stream_t stream) {
    ATVS_CHECK_ARG(a && b && out, ATVS_E_NULL, "atvs_add: NULL pointer");
    if (n <= 0) return 0;
    cudaStream_t st = (cudaStream_t)stream;
    const unsigned grid = grid_for(n, 256, 8);
    if (dtype == ATVS_F32) k_add<float><<<grid, 256, 0, st>>>((const float*)a, (const float*)b, (float*)out, n);
    else if (dtype == ATVS_BF16)
        k_add<__nv_bfloat16><<<grid, 256, 0, st>>>((const __nv_bfloat16*)a, (const __nv_bfloat16*)b, (__nv_bfloat16*)out, n);
    else if (dtype == ATVS_F16)
        k_add<__half><<<grid, 256, 0, st>>>((const __half*)a, (const __half*)b, (__half*)out, n);
    else {
        atvs_set_error("atvs_add: dtype %d", dtype);
        return ATVS_E_DTYPE;
    }
    ATVS_LAUNCH_CHECK();
    return 0;
}

template <int MODE>
static int launch_att(const void* act, const void* x, int N, long long V, int C, int dtype, const float* gmax,
                      float* out, cudaStream_t st, const char* who) {
    ATVS_CHECK_ARG(act && out && (MODE == 1 || x), ATVS_E_NULL, "%s: NULL pointer", who);
    ATVS_CHECK_ARG(N > 0 && N <= ATT_MAXN && V > 0 && C > 0 && C % 4 == 0, ATVS_E_SHAPE, "%s: N=%d V=%lld C=%d", who, N,
                   V, C);
    const unsigned grid = grid_for(V * (C / 4), 256, 8);
    if (dtype == ATVS_F32)
        k_attention<float, MODE><<<grid, 256, 0, st>>>((const float*)act, (const float*)x, N, V, C, gmax, out);
    else if (dtype == ATVS_BF16)
        k_attention<__nv_bfloat16, MODE><<<grid, 256, 0, st>>>((const __nv_bfloat16*)act, (const __nv_bfloat16*)x, N, V,
                                                               C, gmax, out);
    else if (dtype == ATVS_F16)
        k_attention<__half, MODE><<<grid, 256, 0, st>>>((const __half*)act, (const __half*)x, N, V, C, gmax, out);
    else {
        atvs_set_error("%s: dtype %d", who, dtype);
        return ATVS_E_DTYPE;
    }
    ATVS_LAUNCH_CHECK();
    return 0;
}

extern "C" int atvs_attention_combine(const void* act, const void* x, int N, long long V, int C, int dtype, float* out,
                                      atvs_stream_t stream) {
    return launch_att<0>(act, x, N, V, C, dtype, nullptr, out, (cudaStream_t)stream, "atvs_attention_combine");
}

extern "C" int atvs_attention_local_max(const void* act, int N, long long V, int C, int dtype, float* lmax,
                                        atvs_stream_t stream) {
    return launch_att<1>(act, nullptr, N, V, C, dtype, nullptr, lmax, (cudaStream_t)stream, "atvs_attention_local_max");
}

extern "C" int atvs_attention_partial(const void* act, const void* x, int N, long long V, int C, int dtype,
                                      const float* gmax, float* num_den, atvs_stream_t stream) {
    ATVS_CHECK_ARG(gmax, ATVS_E_NULL, "atvs_attention_partial: gmax is NULL");
    return launch_att<2>(act, x, N, V, C, dtype, gmax, num_den, (cudaStream_t)stream, "atvs_attention_partial");
}

extern "C" int atvs_attention_raw(const void* act_raw, int act_dtype, const void* const* x_views, int N, long long V, int C,
                                  int x_dtype, int mode, const float* gmax, float* out, atvs_stream_t stream) {
    ATVS_CHECK_ARG(act_dtype == ATVS_F32 || act_dtype == ATVS_F16, ATVS_E_DTYPE, "atvs_attention_raw: act_dtype %d", act_dtype);
    ATVS_CHECK_ARG(act_raw && out && (mode == 1 || x_views) && (mode != 2 || gmax), ATVS_E_NULL, "atvs_attention_raw: NULL pointer");
    ATVS_CHECK_ARG(N > 0 && N <= ATT_MAXN && V > 0 && C > 0 && C % 8 == 0, ATVS_E_SHAPE, "atvs_attention_raw: N=%d V=%lld C=%d",
                   N, V, C);
    ATVS_CHECK_ARG(mode >= 0 && mode <= 2, ATVS_E_UNSUP, "atvs_attention_raw: mode %d", mode);
    ATVS_CHECK_ARG((((uintptr_t)act_raw | (uintptr_t)gmax | (uintptr_t)out) & 15) == 0, ATVS_E_SHAPE,
                   "atvs_attention_raw: buffers must be 16-byte aligned");
    AttViews xs;
    for (int n = 0; n < ATT_MAXN; ++n) xs.p[n] = nullptr;
    if (mode != 1)
        for (int n = 0; n < N; ++n) {
            ATVS_CHECK_ARG(x_views[n] && ((uintptr_t)x_views[n] & 15) == 0, ATVS_E_NULL,
                           "atvs_attention_raw: view %d is NULL or not 16-byte aligned", n);
            xs.p[n] = x_views[n];
        }
    cudaStream_t st = (cudaStream_t)stream;
#define ATT_RAW_N(T, M, NM)                                                                                   \
    do {                                                                                                      \
        if (act_dtype == ATVS_F16)                                                                            \
            k_attention_raw<T, __half, M, NM><<<grid_resident<k_attention_raw<T, __half, M, NM>>(V * (C / 8), 256), 256, 0, st>>>( \
                (const __half*)act_raw, xs, N, V, C, gmax, out);                                               \
        else                                                                                                  \
            k_attention_raw<T, float, M, NM><<<grid_resident<k_attention_raw<T, float, M, NM>>(V * (C / 8), 256), 256, 0, st>>>(   \
                (const float*)act_raw, xs, N, V, C, gmax, out);                                                \
    } while (0)
    // the per-view logits live in registers: instantiate for the view count (4 sources at cfg2) so that the
    // kernel keeps its occupancy
#define ATT_RAW(T, M)                                                                                         \
    do {                                                                                                      \
        if (N <= 2) ATT_RAW_N(T, M, 2); else if (N <= 4) ATT_RAW_N(T, M, 4); else ATT_RAW_N(T, M, ATT_MAXN);  \
    } while (0)
    if (x_dtype == ATVS_F32 || mode == 1) {
        if (mode == 0) ATT_RAW(float, 0); else if (mode == 1) ATT_RAW(float, 1); else ATT_RAW(float, 2);
    } else if (x_dtype == ATVS_BF16) {
        if (mode == 0) ATT_RAW(__nv_bfloat16, 0); else ATT_RAW(__nv_bfloat16, 2);
    } else if (x_dtype == ATVS_F16) {
        if (mode == 0) ATT_RAW(__half, 0); else ATT_RAW(__half, 2);
    } else {
        atvs_set_error("atvs_attention_raw: x_dtype %d", x_dtype);
        return ATVS_E_DTYPE;
    }
#undef ATT_RAW
#undef ATT_RAW_N
    ATVS_LAUNCH_CHECK();
    return 0;
}

extern "C" int atvs_attention_finish(const float* num_den, long long V, int C, float* out, atvs_stream_t stream) {
    ATVS_CHECK_ARG(num_den && out, ATVS_E_NULL, "atvs_attention_finish: NULL pointer");
    ATVS_CHECK_ARG(V > 0 && C > 0, ATVS_E_SHAPE, "atvs_attention_finish: V=%lld C=%d", V, C);
    k_attention_finish<<<grid_for(V * C, 256, 8), 256, 0, (cudaStream_t)stream>>>(num_den, V, C, out);
    ATVS_LAUNCH_CHECK();
    return 0;
}
