// Encoder stem on the tensor cores (bf16 activations): 7x7 stride-2 pad-3 convolution 3 -> 64 with folded
// BatchNorm + ReLU, TTA views folded into the loader (same contract as stem.cu, which keeps the fp32
// parity mode).
//
// GEMM view per CTA: D[256 pixels][64 couts] = A[256][K] . B[64][K]^T with K ordered (c, r, s') where the
// 7 horizontal taps are padded to s' = 0..7 (weight 0 for s' = 7): K = 3 * 7 * 8 = 168 (+8 zero) = 176.
// With that order the two bf16 of an A fragment a lane needs are the patch pixels [c][2 py + r][2 px + 2t, + 1],
// one aligned 32-bit word, so A is read straight from the bf16 input patch and no im2col matrix is built.
// 8 warps x (2 output rows x 16 pixels x 64 couts) x 11 k-steps of mma.sync.m16n8k16 (bf16 in, fp32 accumulate):
// a warp owns two output rows so one B fragment read from shared memory feeds two MMAs, and the 16 x 16-pixel
// tile copies the 23.5 KB weight tile once per 256 pixels.  Cin = 3 rules out a TMA / tcgen05 formulation (there
// is no dense channel axis to tile); the stem is 0.3 % of the network's FLOPs and was 4 % of its time on the
// packed fp32 pipe.
#include "common.cuh"

namespace eds {

struct StemViews {
    int m[8][6];
};

constexpr int kSmGroups = 22;                              // 21 (c, r) groups of 8 taps + 1 zero group
constexpr int kSmK = kSmGroups * 8;                        // 176
constexpr int kSmPitch = 184;                              // bf16 per B row (conflict-free fragments)

__device__ __forceinline__ void stem_mma_16816(float (&c)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3,
                                               uint32_t b0, uint32_t b1) {
    asm volatile(
        "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
        : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
        : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}

constexpr int kS2TileH = 16, kS2TileW = 16;
constexpr int kS2PatchH = 2 * kS2TileH + 5;                // 37 input rows
constexpr int kS2PatchW = 40;                              // 37 input cols (+3: tap s' = 7 of the last pixel reads col 37)
constexpr int kS2OutPitch = 72;
constexpr size_t kS2SmemBytes = (size_t)(3 * kS2PatchH * kS2PatchW + 64 * kSmPitch + 256 * kS2OutPitch) * 2;

__global__ void __launch_bounds__(256, 2)
stem_conv_mma16_kernel(const float* __restrict__ x, int B, int H, int W, StemViews views,
                       const __nv_bfloat16* __restrict__ w_packed, const float* __restrict__ bias,
                       __nv_bfloat16* __restrict__ y) {
    extern __shared__ __align__(16) uint8_t sm_raw[];
    __nv_bfloat16* s_in = reinterpret_cast<__nv_bfloat16*>(sm_raw);                 // [3][37][40]
    __nv_bfloat16* s_b = s_in + 3 * kS2PatchH * kS2PatchW;                          // [64][184]
    __nv_bfloat16* s_out = s_b + 64 * kSmPitch;                                     // [256][72]
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int Ho = H / 2, Wo = W / 2;
    const int img = blockIdx.z;         // v * B + b
    const int v = img / B, b = img % B;
    const int oy0 = blockIdx.y * kS2TileH, ox0 = blockIdx.x * kS2TileW;

    for (int i = tid; i < 64 * kSmPitch / 8; i += 256)
        reinterpret_cast<uint4*>(s_b)[i] = __ldg(reinterpret_cast<const uint4*>(w_packed) + i);
    const int* m = views.m[v];
    const float* xb = x + (int64_t)b * 3 * H * W;
    for (int i = tid; i < 3 * kS2PatchH * kS2PatchW; i += 256) {
        const int c = i / (kS2PatchH * kS2PatchW);
        const int rem = i - c * (kS2PatchH * kS2PatchW);
        const int py = rem / kS2PatchW, px = rem - py * kS2PatchW;
        const int iy = 2 * oy0 - 3 + py, ix = 2 * ox0 - 3 + px;  // coordinates in the augmented view
        float val = 0.f;
        if (iy >= 0 && iy < H && ix >= 0 && ix < W) {
            const int sy = m[0] * iy + m[1] * ix + m[2];
            const int sx = m[3] * iy + m[4] * ix + m[5];
            val = __ldg(xb + ((int64_t)c * H + sy) * W + sx);
        }
        s_in[i] = __float2bfloat16_rn(val);
    }
    __syncthreads();

    // warp w: output rows 2w, 2w + 1 of the tile (2 x 16 pixels) x 64 couts
    const int g = lane >> 2, t = lane & 3;
    float acc[2][8][4];
#pragma unroll
    for (int mt = 0; mt < 2; ++mt)
#pragma unroll
        for (int nt = 0; nt < 8; ++nt)
#pragma unroll
            for (int i = 0; i < 4; ++i) acc[mt][nt][i] = 0.f;
    // word (2 bf16) view of the patch; this lane's column offset inside a patch row: pixel g, taps 2t, 2t + 1
    const uint32_t* pw = reinterpret_cast<const uint32_t*>(s_in) + g + t;
    const __nv_bfloat16* bp0 = s_b + g * kSmPitch + 2 * t;
#pragma unroll
    for (int ks = 0; ks < kSmK / 16; ++ks) {
        const int g0 = 2 * ks, g1 = 2 * ks + 1;                       // (c, r) groups of the two k halves
        const int c0 = g0 / 7, r0 = g0 - c0 * 7, c1 = g1 / 7, r1 = g1 - c1 * 7;
        uint32_t a[2][4];
#pragma unroll
        for (int mt = 0; mt < 2; ++mt) {
            const int py = 2 * warp + mt;
            const uint32_t* lo = pw + ((c0 * kS2PatchH + 2 * py + r0) * kS2PatchW) / 2;
            a[mt][0] = lo[0];                                         // pixel g
            a[mt][1] = lo[8];                                         // pixel g + 8 (16 patch columns on)
            if (g1 < 21) {
                const uint32_t* hi = pw + ((c1 * kS2PatchH + 2 * py + r1) * kS2PatchW) / 2;
                a[mt][2] = hi[0];
                a[mt][3] = hi[8];
            } else {
                a[mt][2] = a[mt][3] = 0u;                             // the zero group (k >= 168)
            }
        }
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) {
            const __nv_bfloat16* bp = bp0 + nt * 8 * kSmPitch + ks * 16;
            const uint32_t b0 = *reinterpret_cast<const uint32_t*>(bp), b1 = *reinterpret_cast<const uint32_t*>(bp + 8);
            stem_mma_16816(acc[0][nt], a[0][0], a[0][1], a[0][2], a[0][3], b0, b1);
            stem_mma_16816(acc[1][nt], a[1][0], a[1][1], a[1][2], a[1][3], b0, b1);
        }
    }
    // bias + ReLU + bf16 -> staging tile [256][72] -> 16-byte coalesced stores
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) {
        const float2 bb = *reinterpret_cast<const float2*>(bias + nt * 8 + 2 * t);
#pragma unroll
        for (int mt = 0; mt < 2; ++mt)
#pragma unroll
            for (int half = 0; half < 2; ++half) {
                const float v0 = fmaxf(acc[mt][nt][2 * half] + bb.x, 0.f), v1 = fmaxf(acc[mt][nt][2 * half + 1] + bb.y, 0.f);
                *reinterpret_cast<__nv_bfloat162*>(s_out + ((2 * warp + mt) * 16 + g + half * 8) * kS2OutPitch + nt * 8 + 2 * t) =
                    __floats2bfloat162_rn(v0, v1);
            }
    }
    __syncthreads();
    for (int i = tid; i < 256 * 8; i += 256) {
        const int p = i >> 3, ch8 = i & 7;
        const int oy = oy0 + (p >> 4), ox = ox0 + (p & 15);
        if (oy < Ho && ox < Wo)
            *reinterpret_cast<uint4*>(y + (((int64_t)img * Ho + oy) * Wo + ox) * 64 + ch8 * 8) =
                *reinterpret_cast<const uint4*>(s_out + p * kS2OutPitch + ch8 * 8);
    }
}

// w [7][7][3][64] fp32 (cout innermost) -> B[cout][(c*7 + r)*8 + s] bf16, pitch 184, zero for s = 7 / k >= 168
__global__ void stem_pack_kernel(const float* __restrict__ w, __nv_bfloat16* __restrict__ out) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < 64 * kSmPitch; i += gridDim.x * blockDim.x) {
        const int co = i / kSmPitch, k = i - co * kSmPitch;
        const int gq = k >> 3, s = k & 7;
        float val = 0.f;
        if (gq < 21 && s < 7) {
            const int c = gq / 7, r = gq - c * 7;
            val = w[((r * 7 + s) * 3 + c) * 64 + co];
        }
        out[i] = __float2bfloat16_rn(val);
    }
}

// Launcher used by eds_stem_conv7x7s2 (stem.cu) for bf16 outputs; the views were validated there.
int stem_conv_mma_launch(const float* x, int B, int H, int W, int V, const int* maps, const void* w_packed,
                         const float* bias, void* y, cudaStream_t stream) {
    StemViews views;
    for (int v = 0; v < V; ++v)
        for (int q = 0; q < 6; ++q) views.m[v][q] = maps[v * 6 + q];
    static PerDevice once;
    if (int rc = smem_opt_in(once, stem_conv_mma16_kernel, (int)kS2SmemBytes, "stem_conv_mma16")) return rc;
    dim3 grid(ceil_div(W / 2, kS2TileW), ceil_div(H / 2, kS2TileH), B * V);
    stem_conv_mma16_kernel<<<grid, 256, kS2SmemBytes, stream>>>(x, B, H, W, views, (const __nv_bfloat16*)w_packed, bias,
                                                              (__nv_bfloat16*)y);
    return check_launch("stem_conv_mma16_kernel");
}

int stem_pack_launch(const float* w, void* out, cudaStream_t stream) {
    stem_pack_kernel<<<24, 512, 0, stream>>>(w, (__nv_bfloat16*)out);
    return check_launch("stem_pack_kernel");
}

}  // namespace eds
