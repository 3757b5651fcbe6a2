// 3x3 / stride 1 / pad 1 implicit-GEMM convolution for NARROW outputs (Cout <= 128) on sm_100a:
// persistent CTAs, halo-slab operand reuse, double-buffered TMEM accumulators.
//
// Same arithmetic as conv_igemm_sm100.cu (Conv2dReLU of src/main/archs/unetplusplusstar.py:22-63 with the
// eval-mode BatchNorm folded into w / bias); a different data path for the layers the generic
// kernel cannot feed.  With N = Cout <= 128 a 128 x N x 16 MMA lasts <= 64 cycles but consumes a
// 4 KB A tile: loading a fresh 128-pixel A tile per (tap, 64-channel chunk) needs ~120 B/clk/SM from
// L2 and the generic kernel stalls on TMA latency (measured 650-700 TFLOP/s at Cout = 64, 350 at 32,
// 60-120 at 16; profiles/r01_*).  Here one CTA owns a 32 x 8 pixel tile (two M = 128 halves) and,
// per 64-channel chunk, loads THREE slabs of 34 rows x 8 pixels -- the tile shifted by dw = -1, 0, +1
// -- each of which serves the three vertical taps dh = -1, 0, +1 of both halves through the start
// address of the UMMA descriptor (one image row of the slab = 8 pixels x 128 B = exactly one
// 128B-swizzle atom, so every start address stays atom-aligned).  Operand bytes per MMA fall 2.4x
// (A: 9 x 128 rows -> 3 x 136 rows per chunk and half; B shared by both halves).
//
//   warp 0      TMA producer: per (chunk, dw) one A slab [block_k][8][34][1] (out-of-bounds rows /
//               columns zero-filled = the padding) + three B boxes [block_k][Cout] (taps dh of that dw)
//   warp 1      MMA issuer: 2 halves x 3 taps x block_k/16 tcgen05.mma per stage, accumulators
//               D[half] = 128 lanes x Cout columns in TMEM, two accumulator sets (tile t, t+1)
//   warps 2-5   epilogue of tile t (tcgen05.ld -> bias / residual / ReLU -> bf16 -> global) while the
//               MMA warp already runs tile t+1.
// Tiles are walked round-robin (tile = blockIdx.x + i * gridDim.x), grid = min(#tiles, #SMs).
#include "tc_ptx.cuh"
#include <algorithm>
#include <cstring>
#include <mutex>

namespace eds {

constexpr int kHaloThreads = 192;
constexpr int kHaloStagesMax = 8;
constexpr int kTileRows = 32, kTileCols = 8, kSlabRows = kTileRows + 2;

struct HaloParams {
    CUtensorMap a_map;
    CUtensorMap a_map1;     // optional second input (channels C0.. of the concatenated K axis)
    int k_split;            // channel chunks served by a_map
    CUtensorMap b_map;
    const float* bias;
    const __nv_bfloat16* residual;
    __nv_bfloat16* y;
    int C, block_k, k_chunks, bn;
    int N, H, W, relu;
    int tiles_w, tiles_h, total_tiles;
    int stages, atom_bytes, a_slab_bytes, b_tap_bytes, stage_bytes, tmem_cols;
    uint32_t idesc, desc_hi;
};

__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}

__global__ void __launch_bounds__(kHaloThreads, 1)
conv3x3_halo_kernel(const __grid_constant__ HaloParams p) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + (size_t)p.stages * p.stage_bytes);
    uint64_t* empty_bar = full_bar + kHaloStagesMax;
    uint64_t* tmem_full_bar = empty_bar + kHaloStagesMax;     // [2]
    uint64_t* tmem_empty_bar = tmem_full_bar + 2;             // [2]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty_bar + 2);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (warp == 0 && lane == 0) {
        prefetch_tmap(&p.a_map);
        prefetch_tmap(&p.b_map);
        for (int s = 0; s < p.stages; ++s) {
            mbar_init(&full_bar[s], 1);
            mbar_init(&empty_bar[s], 1);
        }
        for (int b = 0; b < 2; ++b) {
            mbar_init(&tmem_full_bar[b], 1);
            mbar_init(&tmem_empty_bar[b], 4);      // one arrival per epilogue warp
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    if (warp == 1) tmem_alloc(tmem_slot, (uint32_t)p.tmem_cols);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    const int iters_per_tile = 3 * p.k_chunks;

    if (warp == 0) {
        if (lane == 0) {
            // ===== TMA producer =====
            int stage = 0;
            uint32_t phase = 0;
            for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x) {
                const int tw = tile % p.tiles_w;
                const int t2 = tile / p.tiles_w;
                const int th = t2 % p.tiles_h;
                const int n = t2 / p.tiles_h;
                const int w0 = tw * kTileCols, h0 = th * kTileRows;
                for (int kc = 0; kc < p.k_chunks; ++kc)
                    for (int dwi = 0; dwi < 3; ++dwi) {
                        mbar_wait(&empty_bar[stage], phase ^ 1u);
                        mbar_arrive_expect_tx(&full_bar[stage],
                                              (uint32_t)((kSlabRows * p.atom_bytes) + 3 * p.bn * p.block_k * 2));
                        uint8_t* sa = smem + (size_t)stage * p.stage_bytes;
                        uint8_t* sb = sa + p.a_slab_bytes;
                        if (kc < p.k_split)
                            tma_load_4d(sa, &p.a_map, &full_bar[stage], kc * p.block_k, w0 + dwi - 1, h0 - 1, n);
                        else
                            tma_load_4d(sa, &p.a_map1, &full_bar[stage], (kc - p.k_split) * p.block_k, w0 + dwi - 1,
                                        h0 - 1, n);
                        for (int dhi = 0; dhi < 3; ++dhi)
                            tma_load_2d(sb + dhi * p.b_tap_bytes, &p.b_map, &full_bar[stage],
                                        (dhi * 3 + dwi) * p.C + kc * p.block_k, 0);
                        if (++stage == p.stages) { stage = 0; phase ^= 1u; }
                    }
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer: the warp stays converged, one elected lane issues =====
        int stage = 0;
        uint32_t phase = 0;
        const uint32_t lo0 = desc_lo(smem_u32(smem));
        const uint32_t stage16 = (uint32_t)p.stage_bytes >> 4, slab16 = (uint32_t)p.a_slab_bytes >> 4;
        const uint32_t atom16 = (uint32_t)p.atom_bytes >> 4, btap16 = (uint32_t)p.b_tap_bytes >> 4;
        const uint32_t dhi_w = p.desc_hi, idesc = p.idesc, bn = (uint32_t)p.bn;
        const int k_steps = p.block_k / 16;
        int t = 0;
        for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x, ++t) {
            const int buf = t & 1;
            mbar_wait(&tmem_empty_bar[buf], (uint32_t)(((t >> 1) & 1) ^ 1));   // epilogue drained this set
            tc_fence_after();
            const uint32_t d0 = tmem_base + (uint32_t)buf * 2u * bn;
            for (int it = 0; it < iters_per_tile; ++it) {
                mbar_wait(&full_bar[stage], phase);
                tc_fence_after();
                if (elect_one()) {
                    const uint32_t a_st = lo0 + (uint32_t)stage * stage16, b_st = a_st + slab16;
                    const uint32_t acc0 = it > 0 ? 1u : 0u;
#pragma unroll
                    for (int m = 0; m < 2; ++m)
#pragma unroll
                        for (int dhi = 0; dhi < 3; ++dhi) {
                            const uint32_t a_lo = a_st + (uint32_t)(m * 16 + dhi) * atom16;
                            const uint32_t b_lo = b_st + (uint32_t)dhi * btap16;
                            const uint32_t d = d0 + (uint32_t)m * bn;
                            if (k_steps == 4) {
                                umma_bf16_lohi(d, a_lo, b_lo, dhi_w, idesc, dhi > 0 ? 1u : acc0);
                                umma_bf16_lohi(d, a_lo + 2, b_lo + 2, dhi_w, idesc, 1u);
                                umma_bf16_lohi(d, a_lo + 4, b_lo + 4, dhi_w, idesc, 1u);
                                umma_bf16_lohi(d, a_lo + 6, b_lo + 6, dhi_w, idesc, 1u);
                            } else if (k_steps == 2) {
                                umma_bf16_lohi(d, a_lo, b_lo, dhi_w, idesc, dhi > 0 ? 1u : acc0);
                                umma_bf16_lohi(d, a_lo + 2, b_lo + 2, dhi_w, idesc, 1u);
                            } else {
                                umma_bf16_lohi(d, a_lo, b_lo, dhi_w, idesc, dhi > 0 ? 1u : acc0);
                            }
                        }
                }
                __syncwarp();
                if (elect_one()) umma_commit(&empty_bar[stage]);
                __syncwarp();
                if (++stage == p.stages) { stage = 0; phase ^= 1u; }
            }
            if (elect_one()) umma_commit(&tmem_full_bar[buf]);
            __syncwarp();
        }
    } else {
        // ===== epilogue: warp q owns TMEM lanes [32q, 32q+32) of both halves =====
        const int q = warp & 3;
        const int ml = q * 32 + lane;                 // pixel within a half: row = ml / 8, col = ml % 8
        const int r = ml >> 3, cpx = ml & 7;
        int t = 0;
        for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x, ++t) {
            const int buf = t & 1;
            const int tw = tile % p.tiles_w;
            const int t2 = tile / p.tiles_w;
            const int th = t2 % p.tiles_h;
            const int n = t2 / p.tiles_h;
            const int ow = tw * kTileCols + cpx;
            mbar_wait(&tmem_full_bar[buf], (uint32_t)((t >> 1) & 1));
            tc_fence_after();
            for (int m = 0; m < 2; ++m) {
                const int oh = th * kTileRows + m * 16 + r;
                const bool valid = ow < p.W && oh < p.H;
                const int64_t off = (((int64_t)n * p.H + oh) * p.W + ow) * p.bn;
                const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(buf * 2 * p.bn + m * p.bn);
                for (int c = 0; c < p.bn; c += 16) {
                    uint32_t rr[16];
                    tmem_ld16(taddr + (uint32_t)c, rr);
                    if (valid) {
                        float v[16];
#pragma unroll
                        for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(rr[i]);
                        if (p.bias) {
                            const float4* b4 = reinterpret_cast<const float4*>(p.bias + c);
#pragma unroll
                            for (int i = 0; i < 4; ++i) {
                                const float4 b = __ldg(b4 + i);
                                v[4 * i] += b.x; v[4 * i + 1] += b.y; v[4 * i + 2] += b.z; v[4 * i + 3] += b.w;
                            }
                        }
                        if (p.residual) {
                            float r0[8], r1[8];
                            Vec8<__nv_bfloat16>::ld(p.residual + off + c, r0);
                            Vec8<__nv_bfloat16>::ld(p.residual + off + c + 8, r1);
#pragma unroll
                            for (int i = 0; i < 8; ++i) { v[i] += r0[i]; v[8 + i] += r1[i]; }
                        }
                        if (p.relu) {
#pragma unroll
                            for (int i = 0; i < 16; ++i) v[i] = fmaxf(v[i], 0.f);
                        }
                        float o0[8], o1[8];
#pragma unroll
                        for (int i = 0; i < 8; ++i) { o0[i] = v[i]; o1[i] = v[8 + i]; }
                        Vec8<__nv_bfloat16>::st(p.y + off + c, o0);
                        Vec8<__nv_bfloat16>::st(p.y + off + c + 8, o1);
                    }
                }
            }
            // this warp's TMEM reads of the set are complete (tcgen05.wait::ld inside tmem_ld16)
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&tmem_empty_bar[buf]);
        }
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem_base, (uint32_t)p.tmem_cols);
}

static PerDevice g_halo_once;             // the shared-memory opt-in belongs to a device's context
static int g_num_sms = 148;

static int halo_init() {
    return g_halo_once.run([](int dev) {
        cudaError_t e = cudaFuncSetAttribute(conv3x3_halo_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
        if (e != cudaSuccess) {
            set_error("conv3x3_halo: cannot opt in to 227 KB shared memory: %s", cudaGetErrorString(e));
            return (int)EDS_ERR_CUDA;
        }
        int sms = 0;
        if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && sms > 0) g_num_sms = sms;
        return (int)EDS_OK;
    });
}

static int pow2_ceil_i(int v) {
    int p = 1;
    while (p < v) p <<= 1;
    return p;
}

}  // namespace eds

using namespace eds;

extern "C" int eds_conv3x3_halo_supported(int C, int Cout, int R, int S, int stride, int pad) {
    return R == 3 && S == 3 && stride == 1 && pad == 1 && C >= 16 && C % 16 == 0 && Cout >= 16 && Cout % 16 == 0 &&
           Cout <= 128;
}

static int halo_launch(const void* x, int C0, const void* x1, int C1, int N, int H, int W, const void* w,
                       const float* bias, int Cout, int relu, const void* residual, void* y, void* stream) {
    const int C = C0 + C1;
    EDS_REQUIRE(x && w && y, "conv3x3_halo: null pointer");
    EDS_REQUIRE(C0 >= 16 && C0 % 16 == 0 && C1 >= 0 && C1 % 16 == 0 && (x1 != nullptr) == (C1 > 0),
                "conv3x3_halo: C0=%d C1=%d must be multiples of 16", C0, C1);
    EDS_REQUIRE((((uintptr_t)x1) & 15) == 0, "conv3x3_halo: pointers must be 16-byte aligned");
    EDS_REQUIRE(N > 0 && H > 0 && W > 0, "conv3x3_halo: bad shape N=%d H=%d W=%d", N, H, W);
    EDS_REQUIRE(eds_conv3x3_halo_supported(C, Cout, 3, 3, 1, 1),
                "conv3x3_halo: C=%d Cout=%d outside the supported range (multiples of 16, Cout <= 128)", C, Cout);
    EDS_REQUIRE((((uintptr_t)x | (uintptr_t)w | (uintptr_t)y | (uintptr_t)residual | (uintptr_t)bias) & 15) == 0,
                "conv3x3_halo: pointers must be 16-byte aligned");
    if (int rc = igemm_init()) return rc;            // driver entry point for the tensor maps
    if (int rc = halo_init()) return rc;

    HaloParams p;
    memset(&p, 0, sizeof(p));
    p.bias = bias;
    p.residual = (const __nv_bfloat16*)residual;
    p.y = (__nv_bfloat16*)y;
    p.C = C;
    p.block_k = ((C0 | C1) % 64 == 0) ? 64 : ((C0 | C1) % 32 == 0 ? 32 : 16);   // divides both inputs
    p.k_chunks = C / p.block_k;
    p.k_split = C0 / p.block_k;
    p.bn = Cout;
    p.N = N; p.H = H; p.W = W; p.relu = relu;
    p.tiles_w = ceil_div(W, kTileCols);
    p.tiles_h = ceil_div(H, kTileRows);
    const int64_t total = (int64_t)p.tiles_w * p.tiles_h * N;
    EDS_REQUIRE(total < (1ll << 31), "conv3x3_halo: too many tiles");
    p.total_tiles = (int)total;

    const CUtensorMapSwizzle swz = p.block_k == 64 ? CU_TENSOR_MAP_SWIZZLE_128B
                                  : p.block_k == 32 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B;
    const uint32_t layout = p.block_k == 64 ? 2u : (p.block_k == 32 ? 4u : 6u);
    p.atom_bytes = 8 * p.block_k * 2;                               // 8 rows (= one image row of the slab)
    const uint32_t sbo = (uint32_t)p.atom_bytes >> 4;
    p.desc_hi = sbo | (1u << 14) | (layout << 29);
    p.idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(p.bn >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
    p.a_slab_bytes = (kSlabRows * p.atom_bytes + 1023) & ~1023;
    p.b_tap_bytes = (p.bn * p.block_k * 2 + 1023) & ~1023;
    p.stage_bytes = p.a_slab_bytes + 3 * p.b_tap_bytes;
    p.stages = std::max(2, std::min(kHaloStagesMax, (200 * 1024) / p.stage_bytes));
    p.tmem_cols = std::max(32, pow2_ceil_i(4 * p.bn));
    const size_t smem = (size_t)p.stages * p.stage_bytes + 1024 + (2 * kHaloStagesMax + 4) * 8 + 16;
    EDS_REQUIRE(smem <= 227 * 1024 && p.tmem_cols <= 512, "conv3x3_halo: tile does not fit (smem %zu, tmem %d)", smem,
                p.tmem_cols);

    {
        cuuint64_t dims[4] = {(cuuint64_t)C0, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)N};
        cuuint64_t strides[3] = {(cuuint64_t)C0 * 2, (cuuint64_t)W * C0 * 2, (cuuint64_t)H * W * C0 * 2};
        cuuint32_t box[4] = {(cuuint32_t)p.block_k, (cuuint32_t)kTileCols, (cuuint32_t)kSlabRows, 1u};
        if (int rc = tmap_encode_bf16(&p.a_map, x, 4, dims, strides, box, swz, "halo input")) return rc;
        p.a_map1 = p.a_map;
    }
    if (x1) {
        cuuint64_t dims[4] = {(cuuint64_t)C1, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)N};
        cuuint64_t strides[3] = {(cuuint64_t)C1 * 2, (cuuint64_t)W * C1 * 2, (cuuint64_t)H * W * C1 * 2};
        cuuint32_t box[4] = {(cuuint32_t)p.block_k, (cuuint32_t)kTileCols, (cuuint32_t)kSlabRows, 1u};
        if (int rc = tmap_encode_bf16(&p.a_map1, x1, 4, dims, strides, box, swz, "halo second input")) return rc;
    }
    {
        cuuint64_t dims[2] = {(cuuint64_t)9 * C, (cuuint64_t)Cout};
        cuuint64_t strides[1] = {(cuuint64_t)9 * C * 2};
        cuuint32_t box[2] = {(cuuint32_t)p.block_k, (cuuint32_t)p.bn};
        if (int rc = tmap_encode_bf16(&p.b_map, w, 2, dims, strides, box, swz, "halo weights")) return rc;
    }
    const int grid = (int)std::min<int64_t>(total, g_num_sms);
    conv3x3_halo_kernel<<<grid, kHaloThreads, smem, as_stream(stream)>>>(p);
    return check_launch("conv3x3_halo_kernel");
}

extern "C" int eds_conv3x3_halo_bf16(const void* x, int N, int H, int W, int C, const void* w, const float* bias,
                                     int Cout, int relu, const void* residual, void* y, void* stream) {
    return halo_launch(x, C, nullptr, 0, N, H, W, w, bias, Cout, relu, residual, y, stream);
}

extern "C" int eds_conv3x3_halo_bf16_2src(const void* x0, int C0, const void* x1, int C1, int N, int H, int W,
                                          const void* w, const float* bias, int Cout, int relu, const void* residual,
                                          void* y, void* stream) {
    EDS_REQUIRE(x1 && C1 > 0, "conv3x3_halo_2src: second input missing");
    return halo_launch(x0, C0, x1, C1, N, H, W, w, bias, Cout, relu, residual, y, stream);
}
