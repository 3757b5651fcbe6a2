// CUDA-core implicit-GEMM convolution (fp32 accumulate) for either activation dtype.
// Same contract as the tcgen05 kernel in conv_igemm_sm100.cu; it exists for the fp32
// parity mode (probability maps within 1e-4 of the reference's fp32 PyTorch path) and
// as the independent cross-check of the tensor-core kernel in tests/.  It is not a
// fallback: the bf16 product path never dispatches here.
#include "common.cuh"
#include <algorithm>

namespace eds {

constexpr int kBM = 64, kBN = 64, kBK = 16;

template <typename T>
__device__ __forceinline__ void ld4(const T* p, float (&v)[4]);
template <>
__device__ __forceinline__ void ld4<float>(const float* p, float (&v)[4]) {
    const float4 a = *reinterpret_cast<const float4*>(p);
    v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w;
}
template <>
__device__ __forceinline__ void ld4<__nv_bfloat16>(const __nv_bfloat16* p, float (&v)[4]) {
    const uint2 raw = *reinterpret_cast<const uint2*>(p);
    const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&raw);
    const float2 a = __bfloat1622float2(h[0]), b = __bfloat1622float2(h[1]);
    v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y;
}

template <typename T>
__global__ void __launch_bounds__(256)
conv_simt_kernel(const T* __restrict__ x, int N, int H, int W, int C, const T* __restrict__ w,
                 const float* __restrict__ bias, int Cout, int R, int S, int stride, int pad, int Ho, int Wo,
                 int relu, const T* __restrict__ residual, T* __restrict__ y) {
    __shared__ __align__(16) float As[kBK][kBM + 4];
    __shared__ __align__(16) float Bs[kBK][kBN + 4];
    const int tid = threadIdx.x;
    const int64_t M = (int64_t)N * Ho * Wo;
    const int64_t m0 = (int64_t)blockIdx.x * kBM;
    const int n0 = blockIdx.y * kBN;
    const int K = R * S * C;

    // loader role: pixel/cout row lr, 4 consecutive k at lk
    const int lr = tid >> 2, lk = (tid & 3) * 4;
    const int64_t lm = m0 + lr;
    int ln_ = 0, loh = 0, low = 0;
    const bool m_ok = lm < M;
    if (m_ok) {
        low = (int)(lm % Wo);
        loh = (int)((lm / Wo) % Ho);
        ln_ = (int)(lm / ((int64_t)Wo * Ho));
    }
    const bool co_ok = n0 + lr < Cout;

    // compute role: 4x4 micro tile
    const int tm = (tid & 15) * 4, tn = (tid >> 4) * 4;
    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

    for (int tap = 0; tap < R * S; ++tap) {
        const int r = tap / S, s = tap % S;
        const int iy = loh * stride - pad + r, ix = low * stride - pad + s;
        const bool a_ok = m_ok && iy >= 0 && iy < H && ix >= 0 && ix < W;
        const T* a_base = x + (((int64_t)ln_ * H + iy) * W + ix) * C;
        const T* b_base = w + (int64_t)(n0 + lr) * K + (int64_t)tap * C;
        for (int c0 = 0; c0 < C; c0 += kBK) {
            float av[4] = {0.f, 0.f, 0.f, 0.f}, bv[4] = {0.f, 0.f, 0.f, 0.f};
            if (a_ok) ld4<T>(a_base + c0 + lk, av);
            if (co_ok) ld4<T>(b_base + c0 + lk, bv);
            __syncthreads();
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                As[lk + q][lr] = av[q];
                Bs[lk + q][lr] = bv[q];
            }
            __syncthreads();
#pragma unroll
            for (int k = 0; k < kBK; ++k) {
                const float4 a4 = *reinterpret_cast<const float4*>(&As[k][tm]);
                const float4 b4 = *reinterpret_cast<const float4*>(&Bs[k][tn]);
                const float a[4] = {a4.x, a4.y, a4.z, a4.w};
                const float b[4] = {b4.x, b4.y, b4.z, b4.w};
#pragma unroll
                for (int i = 0; i < 4; ++i)
#pragma unroll
                    for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
            }
        }
    }

#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int64_t m = m0 + tm + i;
        if (m >= M) continue;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int co = n0 + tn + j;
            if (co >= Cout) continue;
            float v = acc[i][j] + (bias ? bias[co] : 0.f);
            if (residual) v += Elem<T>::ld(residual + m * Cout + co);
            if (relu) v = fmaxf(v, 0.f);
            Elem<T>::st(y + m * Cout + co, v);
        }
    }
}

// Grouped convolution (ResNeXt 3x3, fp32 parity mode): one thread per output element, channel fastest so a warp's
// stores and weight reads are contiguous; the reduction (taps x channels of the group, in that order) is one fp32 fma
// chain.  w: [Cout][R][S][C / groups].
template <typename T>
__global__ void __launch_bounds__(256)
conv_simt_grouped_kernel(const T* __restrict__ x, int N, int H, int W, int C, const T* __restrict__ w,
                         const float* __restrict__ bias, int cpg, int Cout, int R, int S, int stride, int pad, int Ho,
                         int Wo, int relu, const T* __restrict__ residual, T* __restrict__ y) {
    const int64_t total = (int64_t)N * Ho * Wo * Cout;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int co = (int)(i % Cout);
        const int64_t m = i / Cout;
        const int ow = (int)(m % Wo), oh = (int)((m / Wo) % Ho), n = (int)(m / ((int64_t)Wo * Ho));
        const int c0 = (co / (Cout / (C / cpg))) * cpg;        // first input channel of co's group
        const T* wr = w + (int64_t)co * R * S * cpg;
        float acc = 0.f;
        for (int r = 0; r < R; ++r) {
            const int iy = oh * stride - pad + r;
            if (iy < 0 || iy >= H) continue;
            for (int s = 0; s < S; ++s) {
                const int ix = ow * stride - pad + s;
                if (ix < 0 || ix >= W) continue;
                const T* xp = x + (((int64_t)n * H + iy) * W + ix) * C + c0;
                const T* wp = wr + (r * S + s) * cpg;
                for (int c = 0; c < cpg; ++c) acc = fmaf(Elem<T>::ld(xp + c), Elem<T>::ld(wp + c), acc);
            }
        }
        float v = acc + (bias ? bias[co] : 0.f);
        if (residual) v += Elem<T>::ld(residual + i);
        if (relu) v = fmaxf(v, 0.f);
        Elem<T>::st(y + i, v);
    }
}

}  // namespace eds

using namespace eds;

extern "C" int eds_conv2d_simt_grouped(const void* x, int N, int H, int W, int C, const void* w, const float* bias,
                                       int groups, int Cout, int R, int S, int stride, int pad, int relu,
                                       const void* residual, void* y, int dtype, void* stream) {
    EDS_REQUIRE(x && w && y, "conv2d_simt_grouped: null pointer");
    EDS_REQUIRE(N > 0 && H > 0 && W > 0 && C > 0 && Cout > 0, "conv2d_simt_grouped: bad shape");
    EDS_REQUIRE(groups >= 1 && C % groups == 0 && Cout % groups == 0,
                "conv2d_simt_grouped: C=%d and Cout=%d must be multiples of groups=%d", C, Cout, groups);
    EDS_REQUIRE(R >= 1 && S >= 1 && stride >= 1 && pad >= 0, "conv2d_simt_grouped: bad filter geometry");
    const int Ho = (H + 2 * pad - R) / stride + 1, Wo = (W + 2 * pad - S) / stride + 1;
    EDS_REQUIRE(Ho > 0 && Wo > 0, "conv2d_simt_grouped: empty output");
    const int64_t total = (int64_t)N * Ho * Wo * Cout;
    const unsigned grid = (unsigned)std::min<int64_t>(ceil_div64(total, 256), 148 * 16);
    EDS_DISPATCH_DTYPE(dtype, T, (conv_simt_grouped_kernel<T><<<grid, 256, 0, as_stream(stream)>>>(
                                     (const T*)x, N, H, W, C, (const T*)w, bias, C / groups, Cout, R, S, stride, pad,
                                     Ho, Wo, relu, (const T*)residual, (T*)y)));
    return check_launch("conv_simt_grouped_kernel");
}

extern "C" int eds_conv2d_simt(const void* x, int N, int H, int W, int C, const void* w, const float* bias,
                               int Cout, int R, int S, int stride, int pad, int relu, const void* residual,
                               void* y, int dtype, void* stream) {
    EDS_REQUIRE(x && w && y, "conv2d_simt: null pointer");
    EDS_REQUIRE(N > 0 && H > 0 && W > 0 && C > 0 && Cout > 0, "conv2d_simt: bad shape");
    EDS_REQUIRE(C % kBK == 0, "conv2d_simt: C=%d must be a multiple of %d", C, kBK);
    EDS_REQUIRE(R >= 1 && S >= 1 && stride >= 1 && pad >= 0, "conv2d_simt: bad filter geometry");
    const int Ho = (H + 2 * pad - R) / stride + 1, Wo = (W + 2 * pad - S) / stride + 1;
    EDS_REQUIRE(Ho > 0 && Wo > 0, "conv2d_simt: empty output");
    const int64_t M = (int64_t)N * Ho * Wo;
    dim3 grid((unsigned)ceil_div64(M, kBM), ceil_div(Cout, kBN));
    EDS_DISPATCH_DTYPE(dtype, T, (conv_simt_kernel<T><<<grid, 256, 0, as_stream(stream)>>>(
                                     (const T*)x, N, H, W, C, (const T*)w, bias, Cout, R, S, stride, pad, Ho, Wo,
                                     relu, (const T*)residual, (T*)y)));
    return check_launch("conv_simt_kernel");
}
