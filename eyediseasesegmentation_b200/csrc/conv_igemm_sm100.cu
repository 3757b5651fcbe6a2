// Implicit-GEMM convolution for sm_100a: TMA-staged NHWC bf16 tiles, tcgen05.mma with the
// fp32 accumulator in tensor memory, fused bias / residual / ReLU epilogue.
//
// Replaces the cuDNN convolutions behind Conv2dReLU (src/main/archs/unetplusplusstar.py:22-63),
// the SENet / ResNet bottleneck convolutions, the axial block's in/out 1x1 convolutions and
// 3x3 stride-2 shortcut (axial_attention_v2.py:243-255) and the attention projections
// (Conv1d k=1 == 1x1 convolution, axial_attention_v2.py:49-52).  BatchNorm is folded into
// w / bias on the host (eval-mode affine).
//
// GEMM view:  D[M = 128 output pixels][N = block_n couts] += A[M][K] * B[N][K]^T,
//             K = taps * C walked as (tap, 64-channel chunk).
//   A tile : one TMA box [block_k ch][TW][TH][TN] of the NHWC input, shifted by the tap's
//            (dh, dw); out-of-bounds elements are zero-filled by TMA = the conv padding.
//            Rows land 128 B apart with the 128B swizzle = the canonical K-major UMMA layout.
//            Stride-2 convolutions read one of four parity planes of the input (plain strided
//            tensor maps), so every tap is still a dense box.
//   B tile : TMA box [block_k][block_n] of the [Cout][taps*C] weight matrix.
//   D      : 128 TMEM lanes x block_n fp32 columns, two buffers (epilogue of tile t overlaps tile t+1).
//   A second input map can follow the first along K (decoder concat read as two dense maps).
//   Grouped mode (ResNeXt 3x3, 64 % channels-per-group == 0): block_n = block_k = 64 and cout tile n reads only
//            input chunk n, so the K loop is the taps alone; the A box starts at channel n * 64 (a_nt_ch) and B is a
//            block-diagonal [Cout][taps][64] matrix (zeros outside each output channel's group).
// Persistent: grid = min(#tiles, #SMs), the TMA ring runs across tile boundaries.
// Warp roles (320 threads): warp 0 = TMA producer, warp 1 = TMEM allocator + MMA issuer,
// warps 2-9 = epilogue (TMEM -> registers -> bias/residual/ReLU -> bf16 -> swizzled shared memory ->
// one TMA bulk tensor store per 64-channel group).
#include "tc_ptx.cuh"
#include <algorithm>
#include <climits>
#include <cstring>
#include <mutex>

namespace eds {

constexpr int kIgemmThreads = 320;   // TMA warp, MMA warp, 8 epilogue warps
constexpr int kMaxTaps = 9;
constexpr int kMaxStages = 8;
constexpr int kTileM = 128;

struct IgemmParams {
    CUtensorMap a_map[4];
    CUtensorMap a_map1;     // optional second input (channels C0.. of the concatenated K axis), stride 1 only
    int k_split;            // channel chunks served by a_map (== k_chunks when there is one input)
    int a_nt_ch;            // input channels the A box advances per cout tile: 64 in grouped mode, 0 when dense
    CUtensorMap b_map;
    const float* bias;
    const float* gate;      // optional [N][Cout]: y = relu((acc + bias) * gate[n][co] + residual)  (SE scale fused)
    const __nv_bfloat16* residual;
    __nv_bfloat16* y;
    int taps, C, block_k, k_chunks, block_n, n_tiles;
    int tw_log2, th_log2, TW, TH, TN;
    int tiles_w, tiles_h;
    int N, Ho, Wo, Cout, relu;
    CUtensorMap y_map;      // output [Cout][Wo][Ho][N], box [st_ch][TW][TH][TN]
    int total_tiles;        // after y_map: nvcc 12.9 then spills 76 / 96 B (stores / loads) instead of 84 / 112 B
    int st_ch, st_bytes, st_bufs, st_mode;   // epilogue staging: channels per TMA store, bytes per buffer, buffers per half, swizzle mode
    int stages, a_stage_bytes, b_stage_bytes, tmem_cols;
    uint32_t idesc;
    uint32_t desc_hi;  // upper 32 bits of the smem descriptor (SBO, version, swizzle mode)
    int8_t tap_plane[kMaxTaps], tap_dh[kMaxTaps], tap_dw[kMaxTaps];
};

__device__ __forceinline__ void mbar_arrive_cta(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// Persistent: grid = min(#tiles, #SMs); CTA i walks tiles i, i + grid, ... (cout tile fastest, so CTAs
// running side by side share their input tile in L2).  The TMA ring runs across tile boundaries and
// the accumulator is double-buffered in TMEM (2 x block_n columns), so the epilogue of tile t
// overlaps the main loop of tile t + 1 and the per-CTA set-up (barriers, TMEM allocation,
// descriptor prefetch) is paid once per SM instead of once per tile.
__global__ void __launch_bounds__(kIgemmThreads, 1)
conv_igemm_kernel(const __grid_constant__ IgemmParams p) {
    extern __shared__ uint8_t smem_raw[];
    // operand stages need 1024 B alignment for the 128B swizzle atom
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    const int stage_bytes = p.a_stage_bytes + p.b_stage_bytes;
    uint8_t* staging = smem + (size_t)p.stages * stage_bytes;          // [2 halves][st_bufs][st_bytes]
    uint8_t* res_stage = staging + (size_t)2 * p.st_bufs * p.st_bytes; // [2 halves][2][st_bytes] when there is a residual
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(res_stage + (p.residual ? (size_t)4 * p.st_bytes : 0));
    uint64_t* empty_bar = full_bar + kMaxStages;
    uint64_t* tmem_full_bar = empty_bar + kMaxStages;      // [2]
    uint64_t* tmem_empty_bar = tmem_full_bar + 2;          // [2]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty_bar + 2);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int num_k_iters = p.taps * p.k_chunks;

    if (warp == 0 && lane == 0) {
        prefetch_tmap(&p.b_map);
        prefetch_tmap(&p.a_map[0]);
        prefetch_tmap(&p.y_map);
        for (int s = 0; s < p.stages; ++s) {
            mbar_init(&full_bar[s], 1);
            mbar_init(&empty_bar[s], 1);
        }
        for (int b = 0; b < 2; ++b) {
            mbar_init(&tmem_full_bar[b], 1);
            mbar_init(&tmem_empty_bar[b], 8);      // one arrival per epilogue warp
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    if (warp == 1) tmem_alloc(tmem_slot, (uint32_t)p.tmem_cols);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        if (lane == 0) {
            // ===== TMA producer =====
            int stage = 0;
            uint32_t phase = 0;
            for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x) {
                const int n_tile = tile % p.n_tiles;
                int m_tile = tile / p.n_tiles;
                const int tile_w = m_tile % p.tiles_w;
                m_tile /= p.tiles_w;
                const int tile_h = m_tile % p.tiles_h;
                const int tile_n = m_tile / p.tiles_h;
                const int w0 = tile_w * p.TW, h0 = tile_h * p.TH, n0 = tile_n * p.TN;
                for (int it = 0; it < num_k_iters; ++it) {
                    const int tap = it / p.k_chunks, kc = it - tap * p.k_chunks;
                    mbar_wait(&empty_bar[stage], phase ^ 1u);
                    mbar_arrive_expect_tx(&full_bar[stage],
                                          (uint32_t)(kTileM * p.block_k * 2 + p.block_n * p.block_k * 2));
                    uint8_t* sa = smem + (size_t)stage * stage_bytes;
                    uint8_t* sb = sa + p.a_stage_bytes;
                    if (kc < p.k_split)
                        tma_load_4d(sa, &p.a_map[p.tap_plane[tap]], &full_bar[stage], kc * p.block_k + n_tile * p.a_nt_ch,
                                    w0 + p.tap_dw[tap], h0 + p.tap_dh[tap], n0);
                    else
                        tma_load_4d(sa, &p.a_map1, &full_bar[stage], (kc - p.k_split) * p.block_k,
                                    w0 + p.tap_dw[tap], h0 + p.tap_dh[tap], n0);
                    tma_load_2d(sb, &p.b_map, &full_bar[stage], tap * p.C + kc * p.block_k, n_tile * p.block_n);
                    if (++stage == p.stages) { stage = 0; phase ^= 1u; }
                }
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer: the warp stays converged, one elected lane issues =====
        int stage = 0;
        uint32_t phase = 0;
        const int k_steps = p.block_k / 16;
        const uint32_t lo0 = desc_lo(smem_u32(smem));
        const uint32_t stage16 = (uint32_t)stage_bytes >> 4, b16 = (uint32_t)p.a_stage_bytes >> 4;
        const uint32_t dhi = p.desc_hi, idesc = p.idesc;
        int t = 0;
        for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x, ++t) {
            const int buf = t & 1;
            mbar_wait(&tmem_empty_bar[buf], (uint32_t)(((t >> 1) & 1) ^ 1));     // epilogue drained this buffer
            tc_fence_after();
            const uint32_t d = tmem_base + (uint32_t)(buf * p.block_n);
            for (int it = 0; it < num_k_iters; ++it) {
                mbar_wait(&full_bar[stage], phase);
                tc_fence_after();
                if (elect_one()) {
                    const uint32_t a_lo = lo0 + (uint32_t)stage * stage16, b_lo = a_lo + b16;
                    if (k_steps == 4) {
                        umma_bf16_lohi(d, a_lo, b_lo, dhi, idesc, it > 0 ? 1u : 0u);
                        umma_bf16_lohi(d, a_lo + 2, b_lo + 2, dhi, idesc, 1u);
                        umma_bf16_lohi(d, a_lo + 4, b_lo + 4, dhi, idesc, 1u);
                        umma_bf16_lohi(d, a_lo + 6, b_lo + 6, dhi, idesc, 1u);
                    } else if (k_steps == 2) {
                        umma_bf16_lohi(d, a_lo, b_lo, dhi, idesc, it > 0 ? 1u : 0u);
                        umma_bf16_lohi(d, a_lo + 2, b_lo + 2, dhi, idesc, 1u);
                    } else {
                        umma_bf16_lohi(d, a_lo, b_lo, dhi, idesc, it > 0 ? 1u : 0u);
                    }
                    umma_commit(&empty_bar[stage]);  // frees the stage once these MMAs have read it
                }
                __syncwarp();
                if (++stage == p.stages) { stage = 0; phase ^= 1u; }
            }
            if (elect_one()) umma_commit(&tmem_full_bar[buf]);
            __syncwarp();
        }
    } else {
        // ===== epilogue: 8 warps; warp w may only touch TMEM lanes [32 (w % 4), +32), so two warps share
        // a lane quadrant and the two "halves" (4 warps = 128 rows each) take alternate channel groups.
        // A group of st_ch channels of the 128-pixel tile is staged in shared memory in the TMA
        // swizzle and leaves as ONE bulk tensor store (coalesced, clipped at the map edge by TMA).
        const int q = warp & 3;
        const int half = (warp - 2) >> 2;
        const int m = q * 32 + lane;
        const int tw = m & (p.TW - 1);
        const int th = (m >> p.tw_log2) & (p.TH - 1);
        const int tn = m >> (p.tw_log2 + p.th_log2);
        const int n_groups = p.block_n / p.st_ch;
        const int row_bytes = p.st_ch * 2;
        // 16-byte chunk j of row m lives at chunk j ^ swz(m): 128B mode m & 7, 64B (m >> 1) & 3, 32B (m >> 2) & 1
        const uint32_t swz = p.st_mode == 0 ? (uint32_t)(m & 7) : (p.st_mode == 1 ? (uint32_t)((m >> 1) & 3) : (uint32_t)((m >> 2) & 1));
        uint8_t* my_stage = staging + (size_t)half * p.st_bufs * p.st_bytes;
        const bool issuer = (warp - 2) % 4 == 0 && lane == 0;      // first warp of the half
        // Residual (skip connection / SE bottleneck tail): the [128 pixels][st_ch] tile of a group is fetched
        // COOPERATIVELY with cp.async, 16-byte chunk by chunk in row-major order of the staging layout (a warp copies
        // whole 128-byte pixel rows: coalesced), into one of two buffers of this half, ONE GROUP AHEAD of its use.
        // (A lane owns one PIXEL: reading its residual directly touched 32 different lines per load instruction and
        // doubled the time of the SE bottleneck's conv3 once scale + residual + ReLU moved into this epilogue.)
        uint8_t* my_res = res_stage + (size_t)half * 2 * p.st_bytes;
        const int hid = (warp - 2) % 4 * 32 + lane;                // thread index inside the half (0..127)
        auto fetch_residual = [&](int tile_, int grp_, uint8_t* dstbuf) {
            const int cpr = row_bytes >> 4;                         // 16-byte chunks per staging row: 8 / 4 / 2
            const int n_tile_ = tile_ % p.n_tiles;
            int m_tile_ = tile_ / p.n_tiles;
            const int w0_ = (m_tile_ % p.tiles_w) * p.TW;
            m_tile_ /= p.tiles_w;
            const int h0_ = (m_tile_ % p.tiles_h) * p.TH, n0_ = (m_tile_ / p.tiles_h) * p.TN;
            const int64_t c0_ = (int64_t)n_tile_ * p.block_n + grp_ * p.st_ch;
#pragma unroll 1
            for (int qc = hid; qc < kTileM * cpr; qc += 128) {
                const int rr = qc / cpr, jc = qc - rr * cpr;
                const int rw = w0_ + (rr & (p.TW - 1)), rh = h0_ + ((rr >> p.tw_log2) & (p.TH - 1));
                const int rn = n0_ + (rr >> (p.tw_log2 + p.th_log2));
                if (rw < p.Wo && rh < p.Ho && rn < p.N) {
                    const uint32_t sw = p.st_mode == 0 ? (uint32_t)(rr & 7)
                                      : (p.st_mode == 1 ? (uint32_t)((rr >> 1) & 3) : (uint32_t)((rr >> 2) & 1));
                    const __nv_bfloat16* src = p.residual + (((int64_t)rn * p.Ho + rh) * p.Wo + rw) * p.Cout + c0_ + jc * 8;
                    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(
                                     dstbuf + (size_t)rr * row_bytes + (((uint32_t)jc ^ sw) << 4))), "l"(src) : "memory");
                }
            }
        };
        int t = 0, sbuf = 0, gcount = 0;
        if (p.residual) {                                           // prologue: the first group of this half
            if ((int)blockIdx.x < p.total_tiles && half < n_groups) fetch_residual(blockIdx.x, half, my_res);
            asm volatile("cp.async.commit_group;" ::: "memory");
        }
        for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x, ++t) {
            const int buf = t & 1;
            const int n_tile = tile % p.n_tiles;
            int m_tile = tile / p.n_tiles;
            const int tile_w = m_tile % p.tiles_w;
            m_tile /= p.tiles_w;
            const int tile_h = m_tile % p.tiles_h;
            const int tile_n = m_tile / p.tiles_h;
            const int w0 = tile_w * p.TW, h0 = tile_h * p.TH, n0 = tile_n * p.TN;
            const int ow = w0 + tw, oh = h0 + th, on = n0 + tn;
            const bool valid = ow < p.Wo && oh < p.Ho && on < p.N;
            const int co0 = n_tile * p.block_n;
            const int64_t off = (((int64_t)on * p.Ho + oh) * p.Wo + ow) * p.Cout + co0;
            mbar_wait(&tmem_full_bar[buf], (uint32_t)((t >> 1) & 1));
            tc_fence_after();
            const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(buf * p.block_n);
            for (int grp = half; grp < n_groups; grp += 2) {
                uint8_t* sdst = my_stage + (size_t)sbuf * p.st_bytes;
                // all TMEM loads of the group are issued before the single wait
                uint32_t r[4][16];
                const int n16 = p.st_ch >> 4;
#pragma unroll
                for (int i = 0; i < 4; ++i)
                    if (i < n16) tmem_ld16_nowait(taddr + (uint32_t)(grp * p.st_ch + i * 16), r[i]);
                // bias of the group's channels: requested before the waits below so the global-load latency
                // overlaps them (a load after tcgen05.wait::ld stalled every 16-column step on the long scoreboard)
                float4 bv[4][4];
#pragma unroll
                for (int i = 0; i < 4; ++i)
#pragma unroll
                    for (int e = 0; e < 4; ++e)
                        bv[i][e] = (p.bias && i < n16)
                                       ? __ldg(reinterpret_cast<const float4*>(p.bias + co0 + grp * p.st_ch + i * 16) + e)
                                       : make_float4(0.f, 0.f, 0.f, 0.f);
                // the store that last read this staging buffer must have finished reading it
                if (issuer) {
                    if (p.st_bufs == 2) asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(1) : "memory");
                    else asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(0) : "memory");
                }
                asm volatile("bar.sync %0, 128;" ::"r"(1 + half) : "memory");
                // residual tile: the copy of THIS group was issued one group ago (or in the prologue); issue the
                // next group's now so that it flies during this group's work
                const uint8_t* rcur = my_res + (size_t)(gcount & 1) * p.st_bytes;
                if (p.residual) {
                    int ntile = tile, ngrp = grp + 2;
                    if (ngrp >= n_groups) { ntile = tile + gridDim.x; ngrp = half; }
                    if (ntile < p.total_tiles && ngrp < n_groups) fetch_residual(ntile, ngrp, my_res + (size_t)((gcount + 1) & 1) * p.st_bytes);
                    asm volatile("cp.async.commit_group;" ::: "memory");          // (possibly empty) keeps the count uniform
                }
                tmem_ld_wait();
                if (p.residual) {
                    asm volatile("cp.async.wait_group 1;" ::: "memory");           // everything but the prefetch just issued
                    asm volatile("bar.sync %0, 128;" ::"r"(1 + half) : "memory");  // ... of every thread of the half
                }
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    if (i >= n16) break;
                    const int c16 = i * 16;
                    const int c = grp * p.st_ch + c16;
                    float v[16];
#pragma unroll
                    for (int e = 0; e < 16; ++e) v[e] = __uint_as_float(r[i][e]);
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        const float4 bb = bv[i][e];
                        v[4 * e] += bb.x; v[4 * e + 1] += bb.y; v[4 * e + 2] += bb.z; v[4 * e + 3] += bb.w;
                    }
                    if (p.gate && valid) {                     // squeeze-excitation scale of this image's channels
                        const float4* g4 = reinterpret_cast<const float4*>(p.gate + (int64_t)on * p.Cout + co0 + c);
#pragma unroll
                        for (int e = 0; e < 4; ++e) {
                            const float4 gg = __ldg(g4 + e);
                            v[4 * e] *= gg.x; v[4 * e + 1] *= gg.y; v[4 * e + 2] *= gg.z; v[4 * e + 3] *= gg.w;
                        }
                    }
                    if (p.residual) {                          // this lane's own row of the parked residual tile
                        const uint32_t jr = (uint32_t)c16 >> 3;
                        const uint8_t* rrow = rcur + (size_t)m * row_bytes;
                        float r0[8], r1[8];
                        Vec8<__nv_bfloat16>::ld(reinterpret_cast<const __nv_bfloat16*>(rrow + ((jr ^ swz) << 4)), r0);
                        Vec8<__nv_bfloat16>::ld(reinterpret_cast<const __nv_bfloat16*>(rrow + (((jr + 1) ^ swz) << 4)), r1);
#pragma unroll
                        for (int e = 0; e < 8; ++e) { v[e] += r0[e]; v[8 + e] += r1[e]; }
                    }
                    if (p.relu) {
#pragma unroll
                        for (int e = 0; e < 16; ++e) v[e] = fmaxf(v[e], 0.f);
                    }
                    uint4 o0, o1;
                    {
                        __nv_bfloat162* h0p = reinterpret_cast<__nv_bfloat162*>(&o0);
                        __nv_bfloat162* h1p = reinterpret_cast<__nv_bfloat162*>(&o1);
#pragma unroll
                        for (int e = 0; e < 4; ++e) {
                            h0p[e] = __floats2bfloat162_rn(v[2 * e], v[2 * e + 1]);
                            h1p[e] = __floats2bfloat162_rn(v[8 + 2 * e], v[8 + 2 * e + 1]);
                        }
                    }
                    const uint32_t j = (uint32_t)c16 >> 3;          // 16-byte chunk index of the first 8 channels
                    uint8_t* rowp = sdst + (size_t)m * row_bytes;
                    *reinterpret_cast<uint4*>(rowp + ((j ^ swz) << 4)) = o0;
                    *reinterpret_cast<uint4*>(rowp + (((j + 1) ^ swz) << 4)) = o1;
                }
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                asm volatile("bar.sync %0, 128;" ::"r"(1 + half) : "memory");
                if (issuer) {
                    asm volatile(
                        "cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];"
                        ::"l"(&p.y_map), "r"(smem_u32(sdst)), "r"(co0 + grp * p.st_ch), "r"(w0), "r"(h0), "r"(n0)
                        : "memory");
                    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                }
                sbuf = (sbuf + 1) & (p.st_bufs - 1);
                ++gcount;
            }
            // this warp's TMEM reads of the buffer are complete (tcgen05.wait::ld above)
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_cta(&tmem_empty_bar[buf]);
        }
        if (issuer) asm volatile("cp.async.bulk.wait_group %0;" ::"n"(0) : "memory");    // stores complete before exit
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem_base, (uint32_t)p.tmem_cols);
}

// ---- host side -----------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn g_encode = nullptr;
static std::once_flag g_igemm_once;
static int g_igemm_init_rc = EDS_OK;
static int g_num_sms = 148;

static void igemm_init_once() {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres);
    if (e != cudaSuccess || qres != cudaDriverEntryPointSuccess || !fn) {
        set_error("conv_igemm: cuTensorMapEncodeTiled entry point unavailable (%s)",
                  e != cudaSuccess ? cudaGetErrorString(e) : "driver too old");
        g_igemm_init_rc = EDS_ERR_CUDA;
        return;
    }
    g_encode = reinterpret_cast<EncodeTiledFn>(fn);
}

static PerDevice g_igemm_attr_once;       // the shared-memory opt-in belongs to a device's context

// The driver entry point is found once per process, the kernel attribute is set once per device.
int igemm_init() {
    std::call_once(g_igemm_once, igemm_init_once);
    if (g_igemm_init_rc) return g_igemm_init_rc;
    return g_igemm_attr_once.run([](int dev) {
        cudaError_t e = cudaFuncSetAttribute(conv_igemm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
        if (e != cudaSuccess) {
            set_error("conv_igemm: cannot opt in to 227 KB shared memory: %s", cudaGetErrorString(e));
            return (int)EDS_ERR_CUDA;
        }
        int sms = 0;
        if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && sms > 0) g_num_sms = sms;
        return (int)EDS_OK;
    });
}

static int ilog2(int v) {
    int l = 0;
    while ((1 << l) < v) ++l;
    return l;
}
static int pow2_ceil(int v) { return 1 << ilog2(v); }

int tmap_encode_bf16(CUtensorMap* map, const void* base, int rank, const cuuint64_t* dims, const cuuint64_t* strides,
                     const cuuint32_t* box, CUtensorMapSwizzle swz, const char* what) {
    cuuint32_t ones[5] = {1, 1, 1, 1, 1};
    CUresult r = g_encode(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, (cuuint32_t)rank, const_cast<void*>(base), dims,
                          strides, box, ones, CU_TENSOR_MAP_INTERLEAVE_NONE, swz, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        set_error("conv_igemm: cuTensorMapEncodeTiled(%s) failed with CUresult %d", what, (int)r);
        return EDS_ERR_CUDA;
    }
    return EDS_OK;
}

}  // namespace eds

using namespace eds;

// x: [N][H][W][C0]; x1 (optional): [N][H][W][C1] -- the convolution of their channel concatenation
// groups > 1: grouped convolution, w the block-diagonal [Cout][R][S][64] matrix (eds_conv2d_igemm_grouped_supported)
static int igemm_launch(const void* x, int C0, const void* x1, int C1, int N, int H, int W, const void* w,
                        const float* bias, int Cout, int R, int S, int stride, int pad, int relu, const void* residual,
                        void* y, void* stream, const float* gate = nullptr, int groups = 1) {
    const int C = C0 + C1;
    EDS_REQUIRE(x && w && y, "conv2d_igemm: null pointer");
    EDS_REQUIRE(N > 0 && H > 0 && W > 0, "conv2d_igemm: bad shape N=%d H=%d W=%d", N, H, W);
    EDS_REQUIRE(C0 >= 16 && C0 % 16 == 0 && C1 >= 0 && C1 % 16 == 0 && (x1 != nullptr) == (C1 > 0),
                "conv2d_igemm: C0=%d C1=%d must be multiples of 16", C0, C1);
    EDS_REQUIRE(!x1 || stride == 1, "conv2d_igemm: two inputs need stride 1");
    EDS_REQUIRE((((uintptr_t)x1) & 15) == 0, "conv2d_igemm: pointers must be 16-byte aligned");
    EDS_REQUIRE(Cout >= 16 && Cout % 16 == 0, "conv2d_igemm: Cout=%d must be a multiple of 16", Cout);
    EDS_REQUIRE(R == S && (R == 1 || R == 3), "conv2d_igemm: filter %dx%d not supported (1x1, 3x3)", R, S);
    EDS_REQUIRE(stride == 1 || stride == 2, "conv2d_igemm: stride=%d not supported", stride);
    EDS_REQUIRE(pad >= 0 && pad <= R / 2, "conv2d_igemm: pad=%d", pad);
    EDS_REQUIRE((((uintptr_t)x | (uintptr_t)w | (uintptr_t)y | (uintptr_t)residual) & 15) == 0 &&
                    (((uintptr_t)bias) & 15) == 0,
                "conv2d_igemm: pointers must be 16-byte aligned");
    if (int rc = igemm_init()) return rc;
    const int Ho = (H + 2 * pad - R) / stride + 1, Wo = (W + 2 * pad - S) / stride + 1;
    EDS_REQUIRE(Ho > 0 && Wo > 0, "conv2d_igemm: empty output");

    IgemmParams p;
    memset(&p, 0, sizeof(p));
    p.bias = bias;
    p.gate = gate;
    EDS_REQUIRE((((uintptr_t)gate) & 15) == 0, "conv2d_igemm: gate must be 16-byte aligned");
    p.residual = (const __nv_bfloat16*)residual;
    p.y = (__nv_bfloat16*)y;
    p.taps = R * S;
    p.C = C;
    p.block_k = ((C0 | C1) % 64 == 0) ? 64 : ((C0 | C1) % 32 == 0 ? 32 : 16);   // divides both inputs
    p.k_chunks = C / p.block_k;
    p.k_split = C0 / p.block_k;
    // cout tile: the largest multiple of 16 that divides Cout and is <= 256 (two accumulators of
    // block_n fp32 columns fit the 512 columns of TMEM)
    int bn = 256;
    while (bn > 16 && Cout % bn != 0) bn -= 16;
    if (groups > 1) {        // one 64-channel input chunk per 64-channel cout tile; B rows are taps x 64 wide
        p.C = 64;
        p.k_chunks = p.k_split = 1;
        p.a_nt_ch = 64;
        bn = 64;
    }
    const int k_iters = p.taps * p.k_chunks;
    p.block_n = bn;
    p.n_tiles = Cout / bn;
    p.N = N; p.Ho = Ho; p.Wo = Wo; p.Cout = Cout; p.relu = relu;

    // pixel tile TN x TH x TW = 128 minimising the number of tiles (ties -> wider rows)
    int best_tiles = INT32_MAX, best_tw = 8;
    for (int tw = 8; tw <= 128; tw *= 2) {
        const int th = std::min(kTileM / tw, pow2_ceil(Ho));
        const int tn = kTileM / (tw * th);
        const int tiles = ceil_div(Wo, tw) * ceil_div(Ho, th) * ceil_div(N, tn);
        if (tiles <= best_tiles) { best_tiles = tiles; best_tw = tw; }
    }
    p.TW = best_tw;
    p.TH = std::min(kTileM / p.TW, pow2_ceil(Ho));
    p.TN = kTileM / (p.TW * p.TH);
    p.tw_log2 = ilog2(p.TW);
    p.th_log2 = ilog2(p.TH);
    p.tiles_w = ceil_div(Wo, p.TW);
    p.tiles_h = ceil_div(Ho, p.TH);
    const int tiles_n = ceil_div(N, p.TN);
    const int64_t n_ctas = (int64_t)p.tiles_w * p.tiles_h * tiles_n * p.n_tiles;
    EDS_REQUIRE(n_ctas < (1ll << 31), "conv2d_igemm: grid too large");

    const CUtensorMapSwizzle swz = p.block_k == 64 ? CU_TENSOR_MAP_SWIZZLE_128B
                                  : p.block_k == 32 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B;
    const uint32_t layout = p.block_k == 64 ? 2u : (p.block_k == 32 ? 4u : 6u);
    const uint32_t sbo = (uint32_t)(8 * p.block_k * 2) >> 4;
    p.desc_hi = sbo | (1u << 14) | (layout << 29);
    p.idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(p.block_n >> 3) << 17) | ((uint32_t)(kTileM >> 4) << 24);
    p.a_stage_bytes = kTileM * p.block_k * 2;                          // 16 / 8 / 4 KB
    p.b_stage_bytes = (p.block_n * p.block_k * 2 + 1023) & ~1023;
    const int stage_bytes = p.a_stage_bytes + p.b_stage_bytes;
    // epilogue staging: groups of st_ch channels (<= 128 B rows so the TMA swizzle applies)
    p.st_ch = (p.block_n % 64 == 0) ? 64 : (p.block_n % 32 == 0 ? 32 : 16);
    p.st_mode = p.st_ch == 64 ? 0 : (p.st_ch == 32 ? 1 : 2);
    p.st_bytes = kTileM * p.st_ch * 2;                                 // 16 / 8 / 4 KB
    // short reductions are store-bound: overlap the bulk stores with the next groups (st_bufs per half in flight)
    p.st_bufs = k_iters <= 8 ? 2 : 1;
    // one persistent CTA per SM: the rest of the shared memory is one TMA ring
    const int res_bytes = residual ? 4 * p.st_bytes : 0;               // two residual buffers per epilogue half
    // one persistent CTA per SM: the rest of the shared memory is one TMA ring of at least two stages (fewer staging
    // buffers if that is what it takes)
    int ring_budget = 0;
    for (;; p.st_bufs >>= 1) {
        ring_budget = 227 * 1024 - 1024 /*align slack*/ - 512 /*barriers*/ - 2 * p.st_bufs * p.st_bytes - res_bytes;
        if (ring_budget >= 2 * stage_bytes || p.st_bufs == 1) break;
    }
    EDS_REQUIRE(ring_budget >= 2 * stage_bytes, "conv2d_igemm: shared memory budget exhausted (stage %d B)", stage_bytes);
    p.stages = std::min(kMaxStages, ring_budget / stage_bytes);
    p.tmem_cols = std::max(32, pow2_ceil(2 * p.block_n));
    p.total_tiles = (int)n_ctas;
    const size_t smem = (size_t)p.stages * stage_bytes + (size_t)2 * p.st_bufs * p.st_bytes + (size_t)res_bytes +
                        1024 /*align slack*/ +
                        (2 * kMaxStages + 4) * 8 + 16;

    // input tensor maps: one per (row parity, col parity) plane that a tap touches
    bool plane_used[4] = {false, false, false, false};
    for (int r = 0; r < R; ++r)
        for (int s = 0; s < S; ++s) {
            const int t = r * S + s;
            const int qh = r - pad, qw = s - pad;
            if (stride == 1) {
                p.tap_plane[t] = 0; p.tap_dh[t] = (int8_t)qh; p.tap_dw[t] = (int8_t)qw;
            } else {
                const int ph = qh & 1, pw = qw & 1;  // parity (two's complement: -1 & 1 == 1)
                p.tap_plane[t] = (int8_t)(ph * 2 + pw);
                p.tap_dh[t] = (int8_t)((qh - ph) / 2);
                p.tap_dw[t] = (int8_t)((qw - pw) / 2);
            }
            plane_used[p.tap_plane[t]] = true;
        }
    const __nv_bfloat16* xb = (const __nv_bfloat16*)x;
    for (int pl = 0; pl < 4; ++pl) {
        if (!plane_used[pl]) continue;
        const int ph = stride == 1 ? 0 : pl >> 1, pw = stride == 1 ? 0 : pl & 1;
        const int Wp = (W - pw + stride - 1) / stride, Hp = (H - ph + stride - 1) / stride;
        EDS_REQUIRE(Wp > 0 && Hp > 0, "conv2d_igemm: empty parity plane");
        cuuint64_t dims[4] = {(cuuint64_t)C0, (cuuint64_t)Wp, (cuuint64_t)Hp, (cuuint64_t)N};
        cuuint64_t strides[3] = {(cuuint64_t)stride * C0 * 2, (cuuint64_t)stride * W * C0 * 2,
                                 (cuuint64_t)H * W * C0 * 2};
        cuuint32_t box[4] = {(cuuint32_t)p.block_k, (cuuint32_t)p.TW, (cuuint32_t)p.TH, (cuuint32_t)p.TN};
        if (int rc = tmap_encode_bf16(&p.a_map[pl], xb + ((int64_t)ph * W + pw) * C0, 4, dims, strides, box, swz, "input"))
            return rc;
    }
    if (x1) {
        cuuint64_t dims[4] = {(cuuint64_t)C1, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)N};
        cuuint64_t strides[3] = {(cuuint64_t)C1 * 2, (cuuint64_t)W * C1 * 2, (cuuint64_t)H * W * C1 * 2};
        cuuint32_t box[4] = {(cuuint32_t)p.block_k, (cuuint32_t)p.TW, (cuuint32_t)p.TH, (cuuint32_t)p.TN};
        if (int rc = tmap_encode_bf16(&p.a_map1, x1, 4, dims, strides, box, swz, "second input")) return rc;
    } else {
        p.a_map1 = p.a_map[p.tap_plane[0]];
    }
    if (!plane_used[0]) p.a_map[0] = p.a_map[p.tap_plane[0]];  // keep the prefetch target valid
    {
        cuuint64_t dims[2] = {(cuuint64_t)p.taps * p.C, (cuuint64_t)Cout};
        cuuint64_t strides[1] = {(cuuint64_t)p.taps * p.C * 2};
        cuuint32_t box[2] = {(cuuint32_t)p.block_k, (cuuint32_t)p.block_n};
        if (int rc = tmap_encode_bf16(&p.b_map, w, 2, dims, strides, box, swz, "weights")) return rc;
    }
    const unsigned grid = (unsigned)std::min<int64_t>(n_ctas, g_num_sms);
    {
        const CUtensorMapSwizzle yswz = p.st_mode == 0 ? CU_TENSOR_MAP_SWIZZLE_128B
                                       : p.st_mode == 1 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B;
        cuuint64_t dims[4] = {(cuuint64_t)Cout, (cuuint64_t)Wo, (cuuint64_t)Ho, (cuuint64_t)N};
        cuuint64_t strides[3] = {(cuuint64_t)Cout * 2, (cuuint64_t)Wo * Cout * 2, (cuuint64_t)Ho * Wo * Cout * 2};
        cuuint32_t box[4] = {(cuuint32_t)p.st_ch, (cuuint32_t)p.TW, (cuuint32_t)p.TH, (cuuint32_t)p.TN};
        if (int rc = tmap_encode_bf16(&p.y_map, y, 4, dims, strides, box, yswz, "output")) return rc;
    }
    conv_igemm_kernel<<<grid, kIgemmThreads, smem, as_stream(stream)>>>(p);
    return check_launch("conv_igemm_kernel");
}

extern "C" int eds_conv2d_igemm_bf16(const void* x, int N, int H, int W, int C, const void* w, const float* bias,
                                     int Cout, int R, int S, int stride, int pad, int relu, const void* residual,
                                     void* y, void* stream) {
    return igemm_launch(x, C, nullptr, 0, N, H, W, w, bias, Cout, R, S, stride, pad, relu, residual, y, stream);
}

extern "C" int eds_conv2d_igemm_bf16_gated(const void* x, int N, int H, int W, int C, const void* w, const float* bias,
                                           const float* gate, int Cout, int R, int S, int stride, int pad, int relu,
                                           const void* residual, void* y, void* stream) {
    EDS_REQUIRE(gate, "conv2d_igemm_gated: gate missing");
    return igemm_launch(x, C, nullptr, 0, N, H, W, w, bias, Cout, R, S, stride, pad, relu, residual, y, stream, gate);
}

extern "C" int eds_conv2d_igemm_bf16_2src(const void* x0, int C0, const void* x1, int C1, int N, int H, int W,
                                          const void* w, const float* bias, int Cout, int R, int S, int pad, int relu,
                                          const void* residual, void* y, void* stream) {
    EDS_REQUIRE(x1 && C1 > 0, "conv2d_igemm_2src: second input missing");
    return igemm_launch(x0, C0, x1, C1, N, H, W, w, bias, Cout, R, S, 1, pad, relu, residual, y, stream);
}

extern "C" int eds_conv2d_igemm_grouped_supported(int C, int Cout, int groups, int R, int S, int stride) {
    if (groups < 2 || C <= 0 || C % groups != 0 || C != Cout || C % 64 != 0) return 0;
    const int cpg = C / groups;
    return 64 % cpg == 0 && R == S && (R == 1 || R == 3) && (stride == 1 || stride == 2);
}

extern "C" int eds_conv2d_igemm_bf16_grouped(const void* x, int N, int H, int W, int C, const void* w_packed,
                                             const float* bias, int groups, int Cout, int R, int S, int stride, int pad,
                                             int relu, const void* residual, void* y, void* stream) {
    EDS_REQUIRE(groups >= 2 && C > 0 && C % groups == 0 && 64 % (C / groups) == 0,
                "conv2d_igemm_grouped: C=%d groups=%d: the channels per group must divide 64", C, groups);
    EDS_REQUIRE(C == Cout && C % 64 == 0, "conv2d_igemm_grouped: C=%d Cout=%d must be equal multiples of 64", C, Cout);
    EDS_REQUIRE(eds_conv2d_igemm_grouped_supported(C, Cout, groups, R, S, stride),
                "conv2d_igemm_grouped: filter %dx%d stride %d not supported (1x1, 3x3; stride 1, 2)", R, S, stride);
    return igemm_launch(x, C, nullptr, 0, N, H, W, w_packed, bias, Cout, R, S, stride, pad, relu, residual, y, stream,
                        nullptr, groups);
}
