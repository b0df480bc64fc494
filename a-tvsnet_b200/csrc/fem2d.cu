// fem2d.cu - first CUDA path of the 2-D feature extraction module (ResNetDS2SPP, SURVEY.md 8(f) row N1):
//   atvs_conv2d_fp32            <- tf.layers.conv2d / slim.conv2d (network.py:142-215, 570-599): k = 1 | 3, stride, dilation,
//                                  explicit top/left padding (covers TF 'SAME' and the bottleneck's pad + 'VALID'), bias, ReLU
//   atvs_channel_moments        <- the batch statistics of tf.layers.batch_normalization / slim.batch_norm (training)
//   atvs_bn2d_apply             <- (x - mean) * rsqrt(var + eps) [+ beta] [ReLU]
//   atvs_avg_pool_same          <- tf.layers.average_pooling2d 'SAME' (mean over the valid elements)
//   atvs_resize_bilinear_align  <- tf.image.resize_images(bilinear, align_corners=True) on NHWC
// fp32 CUDA-core kernels (register-tiled direct convolution): the PARITY path of this row.  The tensor-core (tcgen05)
// version - channel-chunked taps, dilation, bias/ReLU epilogue - is the next step; see DESIGN.md section 6.
#include "common.cuh"

namespace {

struct Conv2dParams {
    int B, H, W, Cin, Cout, Ho, Wo;
    int stride, rate, pad_t, pad_l, relu;
    int tiles_x, tiles_y;
};

// d0 += a.x * b.x, d1 += a.y * b.y as ONE fma.rn.f32x2 (sm_100 FFMA2)
__device__ __forceinline__ void ffma2(float& d0, float& d1, float2 a, float2 b) {
    unsigned long long d, ua, ub;
    asm("mov.b64 %0, {%1, %2};" : "=l"(d) : "f"(d0), "f"(d1));
    asm("mov.b64 %0, {%1, %2};" : "=l"(ua) : "f"(a.x), "f"(a.y));
    asm("mov.b64 %0, {%1, %2};" : "=l"(ub) : "f"(b.x), "f"(b.y));
    asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(d) : "l"(ua), "l"(ub));
    asm("mov.b64 {%0, %1}, %2;" : "=f"(d0), "=f"(d1) : "l"(d));
}

constexpr int C2_TH = 8, C2_CO = 32, C2_KC = 32;      // tile: 8 rows x (8 * PX) pixels, 32 output channels, 32-channel K steps
constexpr int C2_CT = C2_CO / 4;                        // output channels per thread
constexpr int C2_WPT = C2_KC * C2_CO / 256;             // weights per thread and K step
constexpr int C2_MINB = 3;                              // blocks per SM
constexpr int C2_UNROLL = 8;                            // all 8 four-channel sub-steps of a K step unrolled: 20.7 ms per cfg2 frame (4: 22.3)

// block = 256 threads = 64 pixel groups (PX consecutive x) x 4 groups of 8 output channels; one 8 x (8*PX) pixel tile
// and 32 output channels per block.  Per (tap, 16-channel chunk) the weights [16][32] are staged in shared memory; a
// thread does PX*32 FMAs per PX input float4 loads and 8 weight LDS.128.  PX = 4 for the large maps, PX = 2 when that
// would leave the SMs with about one block each (the 1/4-resolution layers: occupancy 14 % with PX = 4).
// 16 output channels per thread (64 per block: each loaded input pixel feeds twice the FMAs) were measured at cfg2 (5 views
// batched): 23.9 ms per frame against 20.7 with 8 (168 registers: one block per SM).
template <int K, int PX>
__global__ void __launch_bounds__(256, C2_MINB)
k_conv2d_fp32(const float* __restrict__ x, const float* __restrict__ w, const float* __restrict__ bias,
              const Conv2dParams p, float* __restrict__ out) {
    constexpr int CT = C2_CT, CO = C2_CO, WPT = C2_WPT;
    __shared__ __align__(16) float ws[2][C2_KC][CO];         // double buffered: ONE barrier per K step
    const int t = threadIdx.x;
    const int cg = t & 3, q = t >> 2;
    const int qy = q >> 3, qx = q & 7;
    int tile = blockIdx.x;
    const int tx = tile % p.tiles_x;
    tile /= p.tiles_x;
    const int ty = tile % p.tiles_y;
    const int b = tile / p.tiles_y;
    const int co0 = blockIdx.y * CO;
    const int oy = ty * C2_TH + qy;
    const int ox0 = tx * (8 * PX) + qx * PX;
    float acc[PX][CT];
#pragma unroll
    for (int j = 0; j < PX; ++j)
#pragma unroll
        for (int c = 0; c < CT; ++c) acc[j][c] = 0.f;
    const bool vec = (p.Cin & 3) == 0;
    const float* xb = x + (size_t)b * p.H * p.W * p.Cin;
    // flattened (tap, 16-channel chunk) loop; the weights of step it+1 are fetched into registers while step it computes
    const int nch = (p.Cin + C2_KC - 1) / C2_KC;
    const int nit = K * K * nch;
    float wnext[WPT];
    auto fetch = [&](int it) {
        const int tap = it / nch, c0 = (it - tap * nch) * C2_KC;
#pragma unroll
        for (int r = 0; r < WPT; ++r) {
            const int i = t + r * 256;
            const int ci = i / CO, co = i % CO;
            wnext[r] = (c0 + ci < p.Cin && co0 + co < p.Cout) ? __ldg(w + ((size_t)tap * p.Cin + c0 + ci) * p.Cout + co0 + co) : 0.f;
        }
    };
    auto stage = [&](int buf) {
#pragma unroll
        for (int r = 0; r < WPT; ++r) {
            const int i = t + r * 256;
            ws[buf][i / CO][i % CO] = wnext[r];
        }
    };
    fetch(0);
    stage(0);
    __syncthreads();
    for (int it = 0; it < nit; ++it) {
        const int cur = it & 1;
        const int tap = it / nch, c0 = (it - tap * nch) * C2_KC;
        const int ky = tap / K, kx = tap % K;
        const int iy = oy * p.stride - p.pad_t + ky * p.rate;
        const bool yok = oy < p.Ho && iy >= 0 && iy < p.H;
        int ix[PX];
        bool ok[PX];
#pragma unroll
        for (int j = 0; j < PX; ++j) {
            ix[j] = (ox0 + j) * p.stride - p.pad_l + kx * p.rate;
            ok[j] = yok && (ox0 + j) < p.Wo && ix[j] >= 0 && ix[j] < p.W;
        }
        if (it + 1 < nit) fetch(it + 1);       // global -> registers while this step computes
#pragma unroll C2_UNROLL
        for (int c4 = 0; c4 < C2_KC; c4 += 4) {
            if (c0 + c4 >= p.Cin) break;
            float in[PX][4];
#pragma unroll
            for (int j = 0; j < PX; ++j) {
                if (!ok[j]) {
                    in[j][0] = in[j][1] = in[j][2] = in[j][3] = 0.f;
                } else if (vec) {
                    const float4 v = __ldg(reinterpret_cast<const float4*>(xb + ((size_t)iy * p.W + ix[j]) * p.Cin + c0 + c4));
                    in[j][0] = v.x; in[j][1] = v.y; in[j][2] = v.z; in[j][3] = v.w;
                } else {
#pragma unroll
                    for (int cc = 0; cc < 4; ++cc)
                        in[j][cc] = (c0 + c4 + cc < p.Cin) ? __ldg(xb + ((size_t)iy * p.W + ix[j]) * p.Cin + c0 + c4 + cc) : 0.f;
                }
            }
#pragma unroll
            for (int cc = 0; cc < 4; ++cc) {
#pragma unroll
                for (int c8 = 0; c8 < CT; c8 += 8) {
                    const float4 w0 = *reinterpret_cast<const float4*>(&ws[cur][c4 + cc][cg * CT + c8]);
                    const float4 w1 = *reinterpret_cast<const float4*>(&ws[cur][c4 + cc][cg * CT + c8 + 4]);
#pragma unroll
                    for (int j = 0; j < PX; ++j) {
                        // two IEEE FMAs per instruction (FFMA2): same results, half the issue slots
                        const float2 a2 = make_float2(in[j][cc], in[j][cc]);
                        ffma2(acc[j][c8 + 0], acc[j][c8 + 1], a2, make_float2(w0.x, w0.y));
                        ffma2(acc[j][c8 + 2], acc[j][c8 + 3], a2, make_float2(w0.z, w0.w));
                        ffma2(acc[j][c8 + 4], acc[j][c8 + 5], a2, make_float2(w1.x, w1.y));
                        ffma2(acc[j][c8 + 6], acc[j][c8 + 7], a2, make_float2(w1.z, w1.w));
                    }
                }
            }
        }
        if (it + 1 < nit) stage(cur ^ 1);      // the other buffer: its readers passed the barrier of the previous step
        __syncthreads();
    }
    if (oy >= p.Ho) return;
    const int co = co0 + cg * CT;
#pragma unroll
    for (int j = 0; j < PX; ++j) {
        const int ox = ox0 + j;
        if (ox >= p.Wo) continue;
        float* o = out + (((size_t)b * p.Ho + oy) * p.Wo + ox) * p.Cout + co;
#pragma unroll
        for (int c = 0; c < CT; ++c) {
            if (co + c >= p.Cout) break;
            float v = acc[j][c] + (bias ? __ldg(bias + co + c) : 0.f);
            if (p.relu) v = fmaxf(v, 0.f);
            o[c] = v;
        }
    }
}

// per-channel sum and sum of squares of an (count, C) tensor; 256 % C == 0 keeps a thread on one channel
__global__ void __launch_bounds__(256)
k_channel_moments(const float* __restrict__ x, long long count, int C, double* __restrict__ stats) {
    __shared__ double sh[2][256];
    const long long n = count * C;
    const long long stride = (long long)gridDim.x * blockDim.x;
    double s = 0.0, s2 = 0.0;
    const bool fixed = (256 % C) == 0;
    if (fixed) {
        for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
            const double v = (double)x[i];
            s += v;
            s2 += v * v;
        }
        sh[0][threadIdx.x] = s;
        sh[1][threadIdx.x] = s2;
        __syncthreads();
        if (threadIdx.x < C) {
            double a = 0.0, a2 = 0.0;
            for (int k = threadIdx.x; k < 256; k += C) { a += sh[0][k]; a2 += sh[1][k]; }
            atomicAdd(&stats[threadIdx.x], a);
            atomicAdd(&stats[C + threadIdx.x], a2);
        }
    } else {
        for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
            const double v = (double)x[i];
            const int c = (int)(i % C);
            atomicAdd(&stats[c], v);
            atomicAdd(&stats[C + c], v * v);
        }
    }
}

// few channels that do not divide 256 (the 3-channel image in front of the shallow feature net's first BN: the general
// path above issues two fp64 atomics per ELEMENT onto 2 C addresses - 404 us for a 512x640x3 image): a thread walks whole
// pixels and keeps all C running sums, one warp reduction and 2 C atomics per block at the end
template <int CMAX>
__global__ void __launch_bounds__(256)
k_channel_moments_small(const float* __restrict__ x, long long count, int C, double* __restrict__ stats) {
    __shared__ double sh[8][2 * CMAX];
    double s[CMAX], s2[CMAX];
#pragma unroll
    for (int c = 0; c < CMAX; ++c) s[c] = s2[c] = 0.0;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long px = (long long)blockIdx.x * blockDim.x + threadIdx.x; px < count; px += stride) {
        const float* r = x + px * C;
#pragma unroll
        for (int c = 0; c < CMAX; ++c)
            if (c < C) {
                const double v = (double)r[c];
                s[c] += v;
                s2[c] += v * v;
            }
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int c = 0; c < CMAX; ++c) {
#pragma unroll
        for (int off = 16; off >= 1; off >>= 1) {
            s[c] += __shfl_xor_sync(0xffffffffu, s[c], off);
            s2[c] += __shfl_xor_sync(0xffffffffu, s2[c], off);
        }
        if (lane == 0) { sh[warp][c] = s[c]; sh[warp][CMAX + c] = s2[c]; }
    }
    __syncthreads();
    if (threadIdx.x < 2 * CMAX) {
        const int c = threadIdx.x % CMAX, hi = threadIdx.x / CMAX;
        if (c < C) {
            double a = 0.0;
#pragma unroll
            for (int w = 0; w < 8; ++w) a += sh[w][hi * CMAX + c];
            atomicAdd(&stats[hi * C + c], a);
        }
    }
}

template <typename OutT>
__global__ void __launch_bounds__(256)
k_bn2d_apply(const float* __restrict__ x, const double* __restrict__ stats, const float* __restrict__ beta, long long count,
             int C, float eps, int relu, OutT* __restrict__ out) {
    const long long n = count * C;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const int c = (int)(i % C);
        const double mean = stats[c] / (double)count;
        double var = stats[C + c] / (double)count - mean * mean;
        if (var < 0.0) var = 0.0;
        const float inv = (float)(1.0 / sqrt(var + (double)eps));
        float y = x[i] * inv - (float)mean * inv;
        if (beta) y += beta[c];
        if (relu) y = fmaxf(y, 0.f);
        if (sizeof(OutT) == 2) y = fminf(fmaxf(y, -65504.f), 65504.f);      // fp16 output saturates
        out[i] = (OutT)y;
    }
}

__global__ void __launch_bounds__(256)
k_avg_pool_same(const float* __restrict__ x, int B, int H, int W, int C, int k, int s, int pad_t, int pad_l, int Ho, int Wo,
                float* __restrict__ out) {
    const long long n = (long long)B * Ho * Wo * C;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const int c = (int)(i % C);
        long long r = i / C;
        const int ox = (int)(r % Wo);
        r /= Wo;
        const int oy = (int)(r % Ho);
        const int b = (int)(r / Ho);
        const int y0 = max(oy * s - pad_t, 0), y1 = min(oy * s - pad_t + k, H);
        const int x0 = max(ox * s - pad_l, 0), x1 = min(ox * s - pad_l + k, W);
        float acc = 0.f;
        for (int y = y0; y < y1; ++y)
            for (int xx = x0; xx < x1; ++xx) acc += x[(((size_t)b * H + y) * W + xx) * C + c];
        out[i] = acc / (float)((y1 - y0) * (x1 - x0));
    }
}

// the SPP windows are up to 64 x 64 (the whole map) with a handful of outputs: gridDim.y blocks share one output pixel,
// each block splits its part of the window over 256 / C thread groups (consecutive threads = consecutive channels:
// coalesced rows), reduces through shared memory and adds its share to the (pre-zeroed) output
__global__ void __launch_bounds__(256)
k_avg_pool_same_block(const float* __restrict__ x, int H, int W, int C, int k, int s, int pad_t, int pad_l, int Ho, int Wo,
                      float* __restrict__ out) {
    __shared__ float sh[256];
    int o = blockIdx.x;
    const int ox = o % Wo;
    o /= Wo;
    const int oy = o % Ho;
    const int b = o / Ho;
    const int G = 256 / C;
    const int c = threadIdx.x % C, g = threadIdx.x / C;
    const int y0 = max(oy * s - pad_t, 0), y1 = min(oy * s - pad_t + k, H);
    const int x0 = max(ox * s - pad_l, 0), x1 = min(ox * s - pad_l + k, W);
    const int ww = x1 - x0, nwin = (y1 - y0) * ww;
    float acc = 0.f;
    if (g < G)
        for (int i = blockIdx.y * G + g; i < nwin; i += G * gridDim.y) {
            const int y = y0 + i / ww, xx = x0 + i % ww;
            acc += x[(((size_t)b * H + y) * W + xx) * C + c];
        }
    sh[threadIdx.x] = acc;
    __syncthreads();
    if (threadIdx.x < C) {
        float tot = 0.f;
        for (int q = 0; q < G; ++q) tot += sh[q * C + threadIdx.x];
        atomicAdd(&out[(((size_t)b * Ho + oy) * Wo + ox) * C + threadIdx.x], tot / (float)nwin);
    }
}

__global__ void __launch_bounds__(256)
k_resize_bilinear_align(const float* __restrict__ x, int B, int H, int W, int C, int Ho, int Wo, float* __restrict__ out) {
    const long long n = (long long)B * Ho * Wo * C;
    const float sy = Ho > 1 ? __fdiv_rn((float)(H - 1), (float)(Ho - 1)) : 0.f;
    const float sx = Wo > 1 ? __fdiv_rn((float)(W - 1), (float)(Wo - 1)) : 0.f;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const int c = (int)(i % C);
        long long r = i / C;
        const int ox = (int)(r % Wo);
        r /= Wo;
        const int oy = (int)(r % Ho);
        const int b = (int)(r / Ho);
        const float fy_ = __fmul_rn((float)oy, sy), fx_ = __fmul_rn((float)ox, sx);
        const int y0 = (int)floorf(fy_), x0 = (int)floorf(fx_);
        const int y1 = min(y0 + 1, H - 1), x1 = min(x0 + 1, W - 1);
        const float fy = fy_ - (float)y0, fx = fx_ - (float)x0;
        const float* xb = x + (size_t)b * H * W * C + c;
        const float tl = xb[((size_t)y0 * W + x0) * C], tr = xb[((size_t)y0 * W + x1) * C];
        const float bl = xb[((size_t)y1 * W + x0) * C], br = xb[((size_t)y1 * W + x1) * C];
        const float top = __fadd_rn(tl, __fmul_rn(__fsub_rn(tr, tl), fx));
        const float bot = __fadd_rn(bl, __fmul_rn(__fsub_rn(br, bl), fx));
        out[i] = __fadd_rn(top, __fmul_rn(__fsub_rn(bot, top), fy));
    }
}

inline unsigned ew_grid(long long n) {
    long long g = (n + 255) / 256;
    const long long cap = (long long)atvs_num_sms() * 8;
    return (unsigned)(g < 1 ? 1 : (g > cap ? cap : g));
}

}  // namespace

extern "C" int atvs_conv2d_fp32(const float* x, const float* kernel, const float* bias, int B, int H, int W, int Cin, int Cout,
                                int ksize, int stride, int rate, int pad_top, int pad_left, int Ho, int Wo, int relu,
                                float* out, atvs_stream_t stream) {
    ATVS_CHECK_ARG(x && kernel && out, ATVS_E_NULL, "atvs_conv2d_fp32: NULL pointer");
    ATVS_CHECK_ARG(B > 0 && H > 0 && W > 0 && Cin > 0 && Cout > 0 && Ho > 0 && Wo > 0, ATVS_E_SHAPE, "atvs_conv2d_fp32: bad shape");
    ATVS_CHECK_ARG(ksize == 1 || ksize == 3, ATVS_E_UNSUP, "atvs_conv2d_fp32: kernel size %d (1 or 3)", ksize);
    ATVS_CHECK_ARG(stride >= 1 && rate >= 1 && pad_top >= 0 && pad_left >= 0, ATVS_E_UNSUP, "atvs_conv2d_fp32: stride/rate/pad");
    ATVS_CHECK_ARG((Cin & 3) != 0 || ((uintptr_t)x & 15) == 0, ATVS_E_SHAPE, "atvs_conv2d_fp32: x must be 16-byte aligned");
    Conv2dParams p;
    p.B = B; p.H = H; p.W = W; p.Cin = Cin; p.Cout = Cout; p.Ho = Ho; p.Wo = Wo;
    p.stride = stride; p.rate = rate; p.pad_t = pad_top; p.pad_l = pad_left; p.relu = relu;
    p.tiles_y = (Ho + C2_TH - 1) / C2_TH;
    const int slabs = (Cout + C2_CO - 1) / C2_CO;
    // 4 pixels per thread unless that leaves fewer than ~4 blocks per SM
    int px = 4;
    if ((long long)B * ((Wo + 31) / 32) * p.tiles_y * slabs < 3LL * atvs_num_sms()) px = 2;
    p.tiles_x = (Wo + 8 * px - 1) / (8 * px);
    dim3 grid((unsigned)((long long)B * p.tiles_x * p.tiles_y), (unsigned)slabs);
    cudaStream_t st = (cudaStream_t)stream;
    if (ksize == 1 && px == 4) k_conv2d_fp32<1, 4><<<grid, 256, 0, st>>>(x, kernel, bias, p, out);
    else if (ksize == 1) k_conv2d_fp32<1, 2><<<grid, 256, 0, st>>>(x, kernel, bias, p, out);
    else if (px == 4) k_conv2d_fp32<3, 4><<<grid, 256, 0, st>>>(x, kernel, bias, p, out);
    else k_conv2d_fp32<3, 2><<<grid, 256, 0, st>>>(x, kernel, bias, p, out);
    ATVS_LAUNCH_CHECK();
    return 0;
}

extern "C" int atvs_channel_moments(const float* x, long long count, int C, double* stats, atvs_stream_t stream) {
    ATVS_CHECK_ARG(x && stats, ATVS_E_NULL, "atvs_channel_moments: NULL pointer");
    ATVS_CHECK_ARG(count > 0 && C > 0, ATVS_E_SHAPE, "atvs_channel_moments: count=%lld C=%d", count, C);
    unsigned g = ew_grid(count * C);
    if (g > 592) g = 592;          // fp64 atomics per block: keep the tail short
    if (C <= 8 && (256 % C) != 0) {
        unsigned gs = ew_grid(count);
        if (gs > 592) gs = 592;
        k_channel_moments_small<8><<<gs, 256, 0, (cudaStream_t)stream>>>(x, count, C, stats);
    } else {
        k_channel_moments<<<g, 256, 0, (cudaStream_t)stream>>>(x, count, C, stats);
    }
    ATVS_LAUNCH_CHECK();
    return 0;
}

extern "C" int atvs_bn2d_apply(const float* x, const double* stats, const float* beta, long long count, int C, float eps,
                               int relu, void* out, int out_dtype, atvs_stream_t stream) {
    ATVS_CHECK_ARG(x && stats && out, ATVS_E_NULL, "atvs_bn2d_apply: NULL pointer");
    ATVS_CHECK_ARG(count > 0 && C > 0, ATVS_E_SHAPE, "atvs_bn2d_apply: count=%lld C=%d", count, C);
    ATVS_CHECK_ARG(out_dtype == ATVS_F32 || out_dtype == ATVS_F16, ATVS_E_DTYPE, "atvs_bn2d_apply: out_dtype %d (ATVS_F32 | ATVS_F16)", out_dtype);
    if (out_dtype == ATVS_F16)
        k_bn2d_apply<__half><<<ew_grid(count * C), 256, 0, (cudaStream_t)stream>>>(x, stats, beta, count, C, eps, relu, (__half*)out);
    else
        k_bn2d_apply<float><<<ew_grid(count * C), 256, 0, (cudaStream_t)stream>>>(x, stats, beta, count, C, eps, relu, (float*)out);
    ATVS_LAUNCH_CHECK();
    return 0;
}

extern "C" int atvs_avg_pool_same(const float* x, int B, int H, int W, int C, int ksize, int stride, float* out,
                                  atvs_stream_t stream) {
    ATVS_CHECK_ARG(x && out, ATVS_E_NULL, "atvs_avg_pool_same: NULL pointer");
    ATVS_CHECK_ARG(B > 0 && H > 0 && W > 0 && C > 0 && ksize > 0 && stride > 0, ATVS_E_SHAPE, "atvs_avg_pool_same: bad shape");
    const int Ho = (H + stride - 1) / stride, Wo = (W + stride - 1) / stride;
    int th = (Ho - 1) * stride + ksize - H, tw = (Wo - 1) * stride + ksize - W;
    if (th < 0) th = 0;
    if (tw < 0) tw = 0;
    if (C <= 256 && ksize * ksize >= 64) {
        int splits = (ksize * ksize + 255) / 256;          // <= ~128 window pixels per thread group
        if (splits > 64) splits = 64;
        cudaStream_t st = (cudaStream_t)stream;
        ATVS_CUDA(cudaMemsetAsync(out, 0, sizeof(float) * (size_t)B * Ho * Wo * C, st));
        k_avg_pool_same_block<<<dim3((unsigned)((long long)B * Ho * Wo), (unsigned)splits), 256, 0, st>>>(
            x, H, W, C, ksize, stride, th / 2, tw / 2, Ho, Wo, out);
    }
    else
        k_avg_pool_same<<<ew_grid((long long)B * Ho * Wo * C), 256, 0, (cudaStream_t)stream>>>(x, B, H, W, C, ksize, stride,
                                                                                            th / 2, tw / 2, Ho, Wo, out);
    ATVS_LAUNCH_CHECK();
    return 0;
}

extern "C" int atvs_resize_bilinear_align(const float* x, int B, int H, int W, int C, int Ho, int Wo, float* out,
                                          atvs_stream_t stream) {
    ATVS_CHECK_ARG(x && out, ATVS_E_NULL, "atvs_resize_bilinear_align: NULL pointer");
    ATVS_CHECK_ARG(B > 0 && H > 0 && W > 0 && C > 0 && Ho > 0 && Wo > 0, ATVS_E_SHAPE, "atvs_resize_bilinear_align: bad shape");
    k_resize_bilinear_align<<<ew_grid((long long)B * Ho * Wo * C), 256, 0, (cudaStream_t)stream>>>(x, B, H, W, C, Ho, Wo, out);
    ATVS_LAUNCH_CHECK();
    return 0;
}
