// 3x3 / stride 1 / pad 1 convolution for the full-resolution tail of the decoders (Cin = 16, Cout in {16, 32}).
//
// Reference: conv2 (16 -> 16) + BN + ReLU of the last decoder block (x_0_4 of unetplusplusstar.py:239-263 /
// DecoderBlock.forward :151-161; block 4 of smp.Unet).  At 1024^2 such a layer holds a fraction of a percent of the
// network's FLOPs but its input and output are 1.6 GB maps each (48-map batch): it is bound by bytes, and a
// 16-column tcgen05 tile wastes the 128 x N datapath (measured 100 - 240 TFLOP/s in the implicit-GEMM kernels).  Here one CTA owns a 16 x 32 pixel output tile:
//   1. the 18 x 34 input halo tile is copied to shared memory as bf16;
//   2. 8 warps x (2 rows x 32 px) x Cout x (9 taps x 16 channels) as mma.sync.m16n8k16 straight from that tile
//      (im2col is only an address: row = pixel, k = (tap, channel));
//   3. bias + ReLU -> bf16 -> staging tile -> 16-byte coalesced stores.
#include "common.cuh"

namespace eds {

constexpr int kSmallTH = 16, kSmallTW = 32;                  // output tile
constexpr int kSmallHH = kSmallTH + 2, kSmallHW = kSmallTW + 2;
constexpr int kSmallCin = 16;
constexpr int kSmallPS = kSmallCin + 8;                      // bf16 per halo pixel (bank-conflict-free fragments)
constexpr int kSmallKP = 9 * kSmallCin + 8;                  // bf16 per weight row
constexpr size_t kSmallInBytes = (size_t)kSmallHH * kSmallHW * kSmallPS * 2;

__device__ __forceinline__ void small_mma(float (&c)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0,
                                          uint32_t b1) {
    asm volatile(
        "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
        : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
        : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}

// x [N][H][W][16], wgt [COUT][3][3][16] -> y [N][H][W][COUT]
template <int COUT>
__global__ void __launch_bounds__(256)
conv3x3_small_kernel(const __nv_bfloat16* __restrict__ x, int H, int W, const __nv_bfloat16* __restrict__ wgt,
                     const float* __restrict__ bias, int relu, __nv_bfloat16* __restrict__ y) {
    constexpr int CIN = kSmallCin, PS = kSmallPS, KP = kSmallKP, NT = COUT / 8, KC = CIN / 16, V8N = CIN / 8;
    extern __shared__ __align__(16) uint8_t sm_raw[];
    __nv_bfloat16* s_in = reinterpret_cast<__nv_bfloat16*>(sm_raw);                        // [18][34][PS]
    __nv_bfloat16* s_w = reinterpret_cast<__nv_bfloat16*>(sm_raw + ((kSmallInBytes + 15) & ~(size_t)15));   // [COUT][KP]
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int n = blockIdx.z;
    const int oy0 = blockIdx.y * kSmallTH, ox0 = blockIdx.x * kSmallTW;

    // weights [COUT][3][3][CIN] -> rows of KP
    for (int i = tid; i < COUT * 9 * CIN / 8; i += 256) {
        const int co = i / (9 * CIN / 8), r = i - co * (9 * CIN / 8);
        *reinterpret_cast<uint4*>(s_w + co * KP + r * 8) = __ldg(reinterpret_cast<const uint4*>(wgt) + i);
    }
    // halo tile
    for (int i = tid; i < kSmallHH * kSmallHW * V8N; i += 256) {
        const int v8 = i % V8N, pix = i / V8N;
        const int hy = pix / kSmallHW, hx = pix - hy * kSmallHW;
        const int iy = oy0 - 1 + hy, ix = ox0 - 1 + hx;               // coordinates in the conv input (H x W)
        const bool inside = iy >= 0 && iy < H && ix >= 0 && ix < W;   // outside = the convolution's zero padding
        float2 v[4];
        V8<__nv_bfloat16>::ld(x + (((int64_t)n * H + min(max(iy, 0), H - 1)) * W + min(max(ix, 0), W - 1)) * CIN + v8 * 8, v);
        if (!inside) {
#pragma unroll
            for (int q = 0; q < 4; ++q) v[q] = f2(0.f);
        }
        V8<__nv_bfloat16>::st(s_in + pix * PS + v8 * 8, v);
    }
    __syncthreads();

    // warp w: output rows 2w, 2w+1 of the tile = 4 m16 tiles (row, 16-pixel half)
    const int g = lane >> 2, t = lane & 3;
    float acc[4][NT][4];
#pragma unroll
    for (int m = 0; m < 4; ++m)
#pragma unroll
        for (int nt = 0; nt < NT; ++nt)
#pragma unroll
            for (int i = 0; i < 4; ++i) acc[m][nt][i] = 0.f;
#pragma unroll
    for (int tap = 0; tap < 9; ++tap) {
        const int dy = tap / 3, dx = tap - dy * 3;
#pragma unroll
        for (int kc = 0; kc < KC; ++kc) {
            uint32_t b0[NT], b1[NT];
#pragma unroll
            for (int nt = 0; nt < NT; ++nt) {
                const __nv_bfloat16* bp = s_w + (nt * 8 + g) * KP + tap * CIN + kc * 16 + 2 * t;
                b0[nt] = *reinterpret_cast<const uint32_t*>(bp);
                b1[nt] = *reinterpret_cast<const uint32_t*>(bp + 8);
            }
#pragma unroll
            for (int m = 0; m < 4; ++m) {
                const int r = 2 * warp + (m >> 1), c0 = (m & 1) * 16;
                const __nv_bfloat16* ap = s_in + ((r + dy) * kSmallHW + c0 + g + dx) * PS + kc * 16 + 2 * t;
                const uint32_t a0 = *reinterpret_cast<const uint32_t*>(ap);
                const uint32_t a1 = *reinterpret_cast<const uint32_t*>(ap + 8 * PS);
                const uint32_t a2 = *reinterpret_cast<const uint32_t*>(ap + 8);
                const uint32_t a3 = *reinterpret_cast<const uint32_t*>(ap + 8 * PS + 8);
#pragma unroll
                for (int nt = 0; nt < NT; ++nt) small_mma(acc[m][nt], a0, a1, a2, a3, b0[nt], b1[nt]);
            }
        }
    }
    // bias + ReLU + bf16 -> staging [512 px][COUT + 8] in the (now free) input region -> coalesced stores
    __syncthreads();
    constexpr int OP = COUT + 8;
    __nv_bfloat16* s_out = s_in;
#pragma unroll
    for (int nt = 0; nt < NT; ++nt) {
        const float2 bb = bias ? *reinterpret_cast<const float2*>(bias + nt * 8 + 2 * t) : make_float2(0.f, 0.f);
#pragma unroll
        for (int m = 0; m < 4; ++m) {
            const int r = 2 * warp + (m >> 1), c0 = (m & 1) * 16;
#pragma unroll
            for (int half = 0; half < 2; ++half) {
                float v0 = acc[m][nt][2 * half] + bb.x, v1 = acc[m][nt][2 * half + 1] + bb.y;
                if (relu) { v0 = fmaxf(v0, 0.f); v1 = fmaxf(v1, 0.f); }
                *reinterpret_cast<__nv_bfloat162*>(s_out + (r * kSmallTW + c0 + g + half * 8) * OP + nt * 8 + 2 * t) =
                    __floats2bfloat162_rn(v0, v1);
            }
        }
    }
    __syncthreads();
    for (int i = tid; i < kSmallTH * kSmallTW * (COUT / 8); i += 256) {
        const int c8 = i % (COUT / 8), p = i / (COUT / 8);
        const int oy = oy0 + p / kSmallTW, ox = ox0 + p % kSmallTW;
        if (oy < H && ox < W)
            *reinterpret_cast<uint4*>(y + (((int64_t)n * H + oy) * W + ox) * COUT + c8 * 8) =
                *reinterpret_cast<const uint4*>(s_out + p * OP + c8 * 8);
    }
}

template <int COUT>
static int small_launch(const void* x, int N, int H, int W, const void* w, const float* bias, int relu, void* y,
                        cudaStream_t stream) {
    const size_t smem_mma = ((kSmallInBytes + 15) & ~(size_t)15) + (size_t)COUT * kSmallKP * 2;
    const size_t smem_out = (size_t)kSmallTH * kSmallTW * (COUT + 8) * 2;      // staging reuses the same space
    const size_t smem = smem_mma > smem_out ? smem_mma : smem_out;
    static PerDevice once;                    // one flag per template instance and per device
    if (smem > 48 * 1024)
        if (int rc = smem_opt_in(once, conv3x3_small_kernel<COUT>, (int)smem, "conv3x3_small")) return rc;
    dim3 grid(ceil_div(W, kSmallTW), ceil_div(H, kSmallTH), N);
    conv3x3_small_kernel<COUT><<<grid, 256, smem, stream>>>((const __nv_bfloat16*)x, H, W, (const __nv_bfloat16*)w,
                                                            bias, relu, (__nv_bfloat16*)y);
    return check_launch("conv3x3_small_kernel");
}

}  // namespace eds

using namespace eds;

extern "C" int eds_conv3x3_small_supported(int C, int Cout) {
    return C == kSmallCin && (Cout == 16 || Cout == 32);
}

extern "C" int eds_conv3x3_small_bf16(const void* x, int N, int H, int W, int C, const void* w, const float* bias,
                                      int Cout, int relu, void* y, void* stream) {
    EDS_REQUIRE(x && w && y, "conv3x3_small: null pointer");
    EDS_REQUIRE(eds_conv3x3_small_supported(C, Cout), "conv3x3_small: C=%d Cout=%d (C = 16, Cout = 16 / 32 only)", C,
                Cout);
    EDS_REQUIRE(N > 0 && N <= 65535 && H > 0 && W > 0, "conv3x3_small: bad shape");
    EDS_REQUIRE((((uintptr_t)x | (uintptr_t)w | (uintptr_t)y) & 15) == 0 && ((uintptr_t)bias & 15) == 0,
                "conv3x3_small: pointers must be 16-byte aligned");
    cudaStream_t s = as_stream(stream);
    if (Cout == 16) return small_launch<16>(x, N, H, W, w, bias, relu, y, s);
    return small_launch<32>(x, N, H, W, w, bias, relu, y, s);
}
