// 3x3 / stride 1 / pad 1 implicit-GEMM convolution for VERY narrow outputs (Cout <= 64) on sm_100a:
// the three horizontal taps of a kernel row share ONE A operand and run as one tcgen05.mma of N = 3 * Cout.
//
// Same arithmetic as conv_igemm_sm100.cu / conv3x3_halo_sm100.cu (Conv2dReLU of
// src/main/archs/unetplusplusstar.py:22-63 with the eval-mode BatchNorm folded into w / bias).
//
// Why: with N = Cout = 64 a 128 x 64 x 16 MMA reads 4 KB of A and 2 KB of B from shared memory for 32 cycles of
// tensor work; shared memory delivers 128 B/clk, so the instruction cannot retire in less than 48 cycles and the
// halo kernel measures 62 once the TMA writes of its three dw-shifted slabs share the same port
// (profiles/r01_kernels_full.md: tensor pipe 54 % active).  A one-pixel shift cannot be expressed in the start
// address of a swizzled descriptor (an image pixel is one 128-byte row of the 1024-byte swizzle atom), so instead
// of shifting the INPUT by dw, the three dw taps are computed from the SAME input window into three accumulators
//     acc[dw][h][w'] = sum_{dh, c} W[dh][dw][c] * x[h + dh][w'][c]          (w' = slab column)
// by stacking the three weight tiles of a kernel row along N (B = [W[dh][-1] | W[dh][0] | W[dh][+1]], 3 * Cout
// rows), and the OUTPUT is shifted when the accumulators are combined:
//     out[h][w] = acc[-1][h][w - 1] + acc[0][h][w] + acc[+1][h][w + 1].
// One TMEM lane is one pixel and one warp of the epilogue owns one 32-pixel image row of the tile, so the shift
// is a warp shuffle by one lane.  Per 3 taps the MMA now reads A once (4 KB) + 6 KB of B for 96 cycles of tensor
// work, one slab per channel chunk is written instead of three, and the kernel is tensor-bound again.
// The price: a tile is 32 slab columns wide and yields 30 output columns (the two edge lanes only feed their
// neighbours).
//
//   tile        8 rows x 30 output columns = two M = 128 halves of 4 rows x 32 slab columns
//   stage       one 64-channel chunk: A slab [block_k][32][10][1] (rows h0-1 .. h0+8, columns w0-1 .. w0+30,
//               out-of-image = zero fill = the padding) + nine B boxes [block_k][Cout] ordered (dh, dw)
//   warp 0      TMA producer
//   warp 1      MMA issuer: 2 halves x 3 dh x block_k/16 tcgen05.mma (N = 3 * Cout) per stage; the vertical taps
//               move the A start address by whole image rows of the slab (4 swizzle atoms)
//   warps 2-9   epilogue (warps 2-5: half 0, warps 6-9: half 1): tcgen05.ld of the three accumulators,
//               shuffle-combine, bias / residual / ReLU, bf16 store.  Each half has its own full / empty barrier,
//               so the MMAs of the next tile's first half run while the previous tile is still being drained.
//
// Resident weights: when the whole weight tensor (9 * Cout * C bf16) fits next to three A slabs -- the conv2 layers
// of the narrow decoder blocks (64 -> 64, 32 -> 32, 16 -> 16) and 32 -> 16 -- it is loaded ONCE per CTA and the ring
// carries A slabs only: L2 -> SM traffic per tile drops from 114 KB to 40 KB at Cout = 64 and a tile is bounded by
// its 24 MMAs instead of by the weight re-load.
#include "tc_ptx.cuh"
#include <algorithm>
#include <cstring>
#include <mutex>

namespace eds {

constexpr int kWideThreads = 320;
constexpr int kWideStagesMax = 4;
constexpr int kWideRows = 8, kWideSlabCols = 32, kWideOutCols = 30, kWideSlabRows = kWideRows + 2;

struct WideParams {
    CUtensorMap a_map;
    CUtensorMap a_map1;     // optional second input (channels C0.. of the concatenated K axis)
    int k_split;            // channel chunks served by a_map
    CUtensorMap b_map;
    CUtensorMap y_map;      // output rows [Cout][30 px][1][1], 128-byte swizzle (used when `staged`)
    const float* bias;
    const __nv_bfloat16* residual;
    __nv_bfloat16* y;
    int C, block_k, k_chunks, bn;
    int N, H, W, relu;
    int tiles_w, tiles_h, total_tiles;
    int stages, atom_bytes, a_slab_bytes, b_box_bytes, stage_bytes, tmem_cols;
    int b_resident, b_region_bytes;   // weights loaded once per CTA in front of the A ring
    int staged, staging_off;          // epilogue through swizzled shared memory + TMA store (Cout = 64 and room)
    uint32_t idesc, desc_hi;
};

__device__ __forceinline__ void wide_mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}

__global__ void __launch_bounds__(kWideThreads, 1)
conv3x3_wide_kernel(const __grid_constant__ WideParams p) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    uint8_t* ring = smem + p.b_region_bytes;                  // resident weights (if any) sit in front of the ring
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(ring + (size_t)p.stages * p.stage_bytes);
    uint64_t* empty_bar = full_bar + kWideStagesMax;
    uint64_t* tmem_full_bar = empty_bar + kWideStagesMax;     // [2]: one per half
    uint64_t* tmem_empty_bar = tmem_full_bar + 2;             // [2]
    uint64_t* b_bar = tmem_empty_bar + 2;                     // resident weights have landed
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(b_bar + 1);
    // bias in shared memory: a global load per 16-column group costs the epilogue a long-scoreboard stall per group
    // (ncu: the top stall of the single-chunk layers), a broadcast LDS does not
    float* s_bias = reinterpret_cast<float*>(full_bar + 16);        // 128 B behind the first barrier: 16-byte aligned
    if (threadIdx.x < (unsigned)p.bn) s_bias[threadIdx.x] = p.bias ? __ldg(p.bias + threadIdx.x) : 0.f;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (warp == 0 && lane == 0) {
        prefetch_tmap(&p.a_map);
        prefetch_tmap(&p.a_map1);
        prefetch_tmap(&p.b_map);
        for (int s = 0; s < p.stages; ++s) {
            mbar_init(&full_bar[s], 1);
            mbar_init(&empty_bar[s], 1);
        }
        for (int m = 0; m < 2; ++m) {
            mbar_init(&tmem_full_bar[m], 1);
            mbar_init(&tmem_empty_bar[m], 4);      // one arrival per epilogue warp of the half
        }
        mbar_init(b_bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    if (warp == 1) tmem_alloc(tmem_slot, (uint32_t)p.tmem_cols);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    const uint32_t n3 = 3u * (uint32_t)p.bn;

    if (warp == 0) {
        if (lane == 0) {
            // ===== TMA producer =====
            int stage = 0;
            uint32_t phase = 0;
            const uint32_t a_tx = (uint32_t)(kWideSlabRows * 4 * p.atom_bytes), b_tx = (uint32_t)(9 * p.bn * p.block_k * 2);
            const uint32_t tx = p.b_resident ? a_tx : a_tx + b_tx;
            if (p.b_resident) {
                mbar_arrive_expect_tx(b_bar, b_tx * (uint32_t)p.k_chunks);
                for (int kc = 0; kc < p.k_chunks; ++kc)
                    for (int tap = 0; tap < 9; ++tap)
                        tma_load_2d(smem + (size_t)(kc * 9 + tap) * p.b_box_bytes, &p.b_map, b_bar,
                                    tap * p.C + kc * p.block_k, 0);
            }
            for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x) {
                const int tw = tile % p.tiles_w;
                const int t2 = tile / p.tiles_w;
                const int th = t2 % p.tiles_h;
                const int n = t2 / p.tiles_h;
                const int w0 = tw * kWideOutCols, h0 = th * kWideRows;
                for (int kc = 0; kc < p.k_chunks; ++kc) {
                    mbar_wait(&empty_bar[stage], phase ^ 1u);
                    mbar_arrive_expect_tx(&full_bar[stage], tx);
                    uint8_t* sa = ring + (size_t)stage * p.stage_bytes;
                    uint8_t* sb = sa + p.a_slab_bytes;
                    if (kc < p.k_split)
                        tma_load_4d(sa, &p.a_map, &full_bar[stage], kc * p.block_k, w0 - 1, h0 - 1, n);
                    else
                        tma_load_4d(sa, &p.a_map1, &full_bar[stage], (kc - p.k_split) * p.block_k, w0 - 1, h0 - 1, n);
                    if (!p.b_resident)
                        for (int tap = 0; tap < 9; ++tap)
                            tma_load_2d(sb + tap * p.b_box_bytes, &p.b_map, &full_bar[stage], tap * p.C + kc * p.block_k, 0);
                    if (++stage == p.stages) { stage = 0; phase ^= 1u; }
                }
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer: the warp stays converged, one elected lane issues =====
        int stage = 0;
        uint32_t phase = 0;
        const uint32_t lo0 = desc_lo(smem_u32(ring)), blo0 = desc_lo(smem_u32(smem));
        const uint32_t stage16 = (uint32_t)p.stage_bytes >> 4, slab16 = (uint32_t)p.a_slab_bytes >> 4;
        const uint32_t bchunk16 = 9u * ((uint32_t)p.b_box_bytes >> 4);
        if (p.b_resident) mbar_wait(b_bar, 0);
        const uint32_t atom16 = (uint32_t)p.atom_bytes >> 4, brow16 = 3u * ((uint32_t)p.b_box_bytes >> 4);
        const uint32_t dhi_w = p.desc_hi, idesc = p.idesc;
        const int k_steps = p.block_k / 16;
        int t = 0;
        for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x, ++t) {
            const uint32_t empty_parity = (uint32_t)((t & 1) ^ 1);
            for (int kc = 0; kc < p.k_chunks; ++kc) {
                mbar_wait(&full_bar[stage], phase);
                const uint32_t a_st = lo0 + (uint32_t)stage * stage16;
                const uint32_t b_st = p.b_resident ? blo0 + (uint32_t)kc * bchunk16 : a_st + slab16;
#pragma unroll
                for (int m = 0; m < 2; ++m) {
                    if (kc == 0) mbar_wait(&tmem_empty_bar[m], empty_parity);   // the epilogue drained this half
                    tc_fence_after();
                    if (elect_one()) {
                        const uint32_t d = tmem_base + (uint32_t)m * n3;
#pragma unroll
                        for (int dhi = 0; dhi < 3; ++dhi) {
                            const uint32_t a_lo = a_st + (uint32_t)(m * 16 + dhi * 4) * atom16;
                            const uint32_t b_lo = b_st + (uint32_t)dhi * brow16;
                            for (int ks = 0; ks < k_steps; ++ks)
                                umma_bf16_lohi(d, a_lo + 2u * ks, b_lo + 2u * ks, dhi_w, idesc,
                                               (kc > 0 || dhi > 0 || ks > 0) ? 1u : 0u);
                        }
                    }
                    __syncwarp();
                    if (kc == p.k_chunks - 1) {
                        if (elect_one()) umma_commit(&tmem_full_bar[m]);
                        __syncwarp();
                    }
                }
                if (elect_one()) umma_commit(&empty_bar[stage]);
                __syncwarp();
                if (++stage == p.stages) { stage = 0; phase ^= 1u; }
            }
        }
    } else {
        // ===== epilogue: warp q owns TMEM lanes [32q, 32q+32) = image row q of its half; lane = slab column =====
        const int q = warp & 3;
        const int m = (warp - 2) >> 2;                // warps 2-5 drain half 0, warps 6-9 half 1
        const int bn = p.bn;
        // staged stores: a lane holds one pixel = one 128-byte output row; written directly, every 16-byte store of
        // a warp touches 32 different lines.  Through a swizzled 4 KB buffer per warp the row of 30 pixels leaves as
        // one bulk tensor store (clipped at the map edge by the tensor map).
        uint8_t* stg = smem + p.staging_off + (size_t)(warp - 2) * 4096;
        const int pos = lane - 1;                      // staging row of this lane's pixel
        int t = 0;
        for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x, ++t) {
            const int tw = tile % p.tiles_w;
            const int t2 = tile / p.tiles_w;
            const int th = t2 % p.tiles_h;
            const int n = t2 / p.tiles_h;
            const int ow = tw * kWideOutCols - 1 + lane;
            const bool col_ok = lane >= 1 && lane <= kWideOutCols && ow < p.W;
            {
                mbar_wait(&tmem_full_bar[m], (uint32_t)(t & 1));
                tc_fence_after();
                const int oh = th * kWideRows + m * 4 + q;
                const bool valid = col_ok && oh < p.H;
                const int64_t off = (((int64_t)n * p.H + oh) * p.W + ow) * bn;
                const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)m * n3;
                if (p.staged) {                        // the previous store of this warp has finished reading `stg`
                    if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
                    __syncwarp();
                }
                for (int c = 0; c < bn; c += 16) {
                    uint32_t rl[16], rc[16], rr[16];
                    tmem_ld16_nowait(taddr + (uint32_t)c, rl);                 // dw = -1: wanted by lane + 1
                    tmem_ld16_nowait(taddr + (uint32_t)(bn + c), rc);          // dw =  0
                    tmem_ld16_nowait(taddr + (uint32_t)(2 * bn + c), rr);      // dw = +1: wanted by lane - 1
                    tmem_ld_wait();
                    float v[16];
#pragma unroll
                    for (int i = 0; i < 16; ++i) {
                        const float l = __shfl_up_sync(0xffffffffu, __uint_as_float(rl[i]), 1);
                        const float r = __shfl_down_sync(0xffffffffu, __uint_as_float(rr[i]), 1);
                        v[i] = (l + __uint_as_float(rc[i])) + r;
                    }
                    if (valid || (p.staged && pos >= 0 && pos < kWideOutCols)) {
                        {
                            const float4* b4 = reinterpret_cast<const float4*>(s_bias + c);
#pragma unroll
                            for (int i = 0; i < 4; ++i) {
                                const float4 b = b4[i];
                                v[4 * i] += b.x; v[4 * i + 1] += b.y; v[4 * i + 2] += b.z; v[4 * i + 3] += b.w;
                            }
                        }
                        if (p.residual && valid) {
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
                        if (p.staged) {
                            const uint32_t j = (uint32_t)c >> 3, sw = (uint32_t)pos & 7u;
                            Vec8<__nv_bfloat16>::st(reinterpret_cast<__nv_bfloat16*>(stg + pos * 128 + ((j ^ sw) << 4)), o0);
                            Vec8<__nv_bfloat16>::st(reinterpret_cast<__nv_bfloat16*>(stg + pos * 128 + (((j + 1) ^ sw) << 4)), o1);
                        } else {
                            Vec8<__nv_bfloat16>::st(p.y + off + c, o0);
                            Vec8<__nv_bfloat16>::st(p.y + off + c + 8, o1);
                        }
                    }
                }
                if (p.staged) {
                    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                    __syncwarp();
                    if (lane == 0 && oh < p.H) {
                        asm volatile(
                            "cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];"
                            ::"l"(&p.y_map), "r"(smem_u32(stg)), "r"(0), "r"(tw * kWideOutCols), "r"(oh), "r"(n)
                            : "memory");
                        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                    }
                }
                // this warp's TMEM reads of the half are complete (tcgen05.wait::ld above)
                tc_fence_before();
                __syncwarp();
                if (lane == 0) wide_mbar_arrive(&tmem_empty_bar[m]);
            }
        }
        if (p.staged && lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");   // stores done before exit
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem_base, (uint32_t)p.tmem_cols);
}

static PerDevice g_wide_once;             // the shared-memory opt-in belongs to a device's context
static int g_wide_sms = 148;

static int wide_init() {
    return g_wide_once.run([](int dev) {
        cudaError_t e = cudaFuncSetAttribute(conv3x3_wide_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
        if (e != cudaSuccess) {
            set_error("conv3x3_wide: cannot opt in to 227 KB shared memory: %s", cudaGetErrorString(e));
            return (int)EDS_ERR_CUDA;
        }
        int sms = 0;
        if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && sms > 0) g_wide_sms = sms;
        return (int)EDS_OK;
    });
}

}  // namespace eds

using namespace eds;

extern "C" int eds_conv3x3_wide_supported(int C, int Cout, int R, int S, int stride, int pad) {
    return R == 3 && S == 3 && stride == 1 && pad == 1 && C >= 16 && C % 16 == 0 && Cout >= 16 && Cout % 16 == 0 &&
           Cout <= 64;
}

static int wide_launch(const void* x, int C0, const void* x1, int C1, int N, int H, int W, const void* w,
                       const float* bias, int Cout, int relu, const void* residual, void* y, void* stream) {
    const int C = C0 + C1;
    EDS_REQUIRE(x && w && y, "conv3x3_wide: null pointer");
    EDS_REQUIRE(C0 >= 16 && C0 % 16 == 0 && C1 >= 0 && C1 % 16 == 0 && (x1 != nullptr) == (C1 > 0),
                "conv3x3_wide: C0=%d C1=%d must be multiples of 16", C0, C1);
    EDS_REQUIRE(N > 0 && H > 0 && W > 0, "conv3x3_wide: bad shape N=%d H=%d W=%d", N, H, W);
    EDS_REQUIRE(eds_conv3x3_wide_supported(C, Cout, 3, 3, 1, 1),
                "conv3x3_wide: C=%d Cout=%d outside the supported range (multiples of 16, Cout <= 64)", C, Cout);
    EDS_REQUIRE((((uintptr_t)x | (uintptr_t)x1 | (uintptr_t)w | (uintptr_t)y | (uintptr_t)residual | (uintptr_t)bias) &
                 15) == 0, "conv3x3_wide: pointers must be 16-byte aligned");
    if (int rc = igemm_init()) return rc;            // driver entry point for the tensor maps
    if (int rc = wide_init()) return rc;

    WideParams p;
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
    p.tiles_w = ceil_div(W, kWideOutCols);
    p.tiles_h = ceil_div(H, kWideRows);
    const int64_t total = (int64_t)p.tiles_w * p.tiles_h * N;
    EDS_REQUIRE(total < (1ll << 31), "conv3x3_wide: too many tiles");
    p.total_tiles = (int)total;

    const CUtensorMapSwizzle swz = p.block_k == 64 ? CU_TENSOR_MAP_SWIZZLE_128B
                                  : p.block_k == 32 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B;
    const uint32_t layout = p.block_k == 64 ? 2u : (p.block_k == 32 ? 4u : 6u);
    p.atom_bytes = 8 * p.block_k * 2;                               // 8 pixels; one image row of the slab = 4 atoms
    const uint32_t sbo = (uint32_t)p.atom_bytes >> 4;
    p.desc_hi = sbo | (1u << 14) | (layout << 29);
    p.idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)((3 * p.bn) >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
    p.a_slab_bytes = (kWideSlabRows * 4 * p.atom_bytes + 1023) & ~1023;
    p.b_box_bytes = p.bn * p.block_k * 2;                           // bn rows, contiguous: the 3 boxes of a kernel row
    const int barrier_bytes = 128 + 64 * 4;   // 13 barriers + TMEM slot in the first 128 B, then the bias
    const int budget = 227 * 1024 - 1024 - barrier_bytes;
    const int b_all = p.k_chunks * 9 * p.b_box_bytes;               // the whole weight tensor
    p.b_resident = b_all + 3 * p.a_slab_bytes <= budget;
    p.b_region_bytes = p.b_resident ? ((b_all + 1023) & ~1023) : 0;
    // the 9 boxes of a chunk are contiguous: the 3 of a kernel row stack into one [3 * bn][block_k] operand
    p.stage_bytes = p.b_resident ? p.a_slab_bytes : ((p.a_slab_bytes + 9 * p.b_box_bytes + 1023) & ~1023);
    p.stages = std::min(kWideStagesMax, (budget - p.b_region_bytes) / p.stage_bytes);
    EDS_REQUIRE(p.stages >= 2, "conv3x3_wide: a stage of %d B leaves no room for double buffering", p.stage_bytes);
    int cols = 32;
    while (cols < 6 * p.bn) cols <<= 1;
    p.tmem_cols = cols;
    // staged epilogue when 8 x 4 KB fit behind the ring (the resident-weight 64 -> 64 layers; the multi-chunk layers
    // hide their epilogue behind the MMAs of the next tile and need the room for the second stage).
    // layout: [weights][ring][barriers + bias (barrier_bytes)][pad to 1024][staging]
    const int after_bars = p.b_region_bytes + p.stages * p.stage_bytes + barrier_bytes;
    p.staging_off = (after_bars + 1023) & ~1023;
    p.staged = p.bn == 64 && p.block_k == 64 && p.staging_off + 8 * 4096 + 1024 <= 227 * 1024;
    const size_t smem = (p.staged ? (size_t)p.staging_off + 8 * 4096 : (size_t)after_bars) + 1024;
    EDS_REQUIRE(smem <= 227 * 1024 && p.tmem_cols <= 512, "conv3x3_wide: tile does not fit (smem %zu, tmem %d)", smem,
                p.tmem_cols);

    {
        cuuint64_t dims[4] = {(cuuint64_t)C0, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)N};
        cuuint64_t strides[3] = {(cuuint64_t)C0 * 2, (cuuint64_t)W * C0 * 2, (cuuint64_t)H * W * C0 * 2};
        cuuint32_t box[4] = {(cuuint32_t)p.block_k, (cuuint32_t)kWideSlabCols, (cuuint32_t)kWideSlabRows, 1u};
        if (int rc = tmap_encode_bf16(&p.a_map, x, 4, dims, strides, box, swz, "wide input")) return rc;
        p.a_map1 = p.a_map;
    }
    if (x1) {
        cuuint64_t dims[4] = {(cuuint64_t)C1, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)N};
        cuuint64_t strides[3] = {(cuuint64_t)C1 * 2, (cuuint64_t)W * C1 * 2, (cuuint64_t)H * W * C1 * 2};
        cuuint32_t box[4] = {(cuuint32_t)p.block_k, (cuuint32_t)kWideSlabCols, (cuuint32_t)kWideSlabRows, 1u};
        if (int rc = tmap_encode_bf16(&p.a_map1, x1, 4, dims, strides, box, swz, "wide second input")) return rc;
    }
    {
        cuuint64_t dims[2] = {(cuuint64_t)9 * C, (cuuint64_t)Cout};
        cuuint64_t strides[1] = {(cuuint64_t)9 * C * 2};
        cuuint32_t box[2] = {(cuuint32_t)p.block_k, (cuuint32_t)p.bn};
        if (int rc = tmap_encode_bf16(&p.b_map, w, 2, dims, strides, box, swz, "wide weights")) return rc;
    }
    if (p.staged) {
        cuuint64_t dims[4] = {(cuuint64_t)Cout, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)N};
        cuuint64_t strides[3] = {(cuuint64_t)Cout * 2, (cuuint64_t)W * Cout * 2, (cuuint64_t)H * W * Cout * 2};
        cuuint32_t box[4] = {64u, (cuuint32_t)kWideOutCols, 1u, 1u};
        if (int rc = tmap_encode_bf16(&p.y_map, y, 4, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B, "wide output")) return rc;
    }
    const int grid = (int)std::min<int64_t>(total, g_wide_sms);
    conv3x3_wide_kernel<<<grid, kWideThreads, smem, as_stream(stream)>>>(p);
    return check_launch("conv3x3_wide_kernel");
}

extern "C" int eds_conv3x3_wide_bf16(const void* x, int N, int H, int W, int C, const void* w, const float* bias,
                                     int Cout, int relu, const void* residual, void* y, void* stream) {
    return wide_launch(x, C, nullptr, 0, N, H, W, w, bias, Cout, relu, residual, y, stream);
}

extern "C" int eds_conv3x3_wide_bf16_2src(const void* x0, int C0, const void* x1, int C1, int N, int H, int W,
                                          const void* w, const float* bias, int Cout, int relu, const void* residual,
                                          void* y, void* stream) {
    EDS_REQUIRE(x1 && C1 > 0, "conv3x3_wide_2src: second input missing");
    return wide_launch(x0, C0, x1, C1, N, H, W, w, bias, Cout, relu, residual, y, stream);
}
