// Decoder concat + SCSE with DEFERRED gates: the gated map is never written twice.
//
// Reference: DecoderBlock.forward (src/main/archs/unetplusplusstar.py:151-161; smp SCSEModule, 3P):
//     x = cat([interpolate(x, 2), *skips]); x = attention1(x); x = conv1(x); x = conv2(x); x = attention2(x)
// SCSE scales every element by cSE[n][c] + sSE[n][p]; both need a global pass over the map first
// (channel means, per-pixel w_sse . x).  Instead of materialising a map and then re-writing it
// scaled (4 full passes per concat in the first version, see scse.cu), a map carries its gate as
// two small side tensors until somebody reads it:
//
//     value[n][p][c] = x[n][p][c] * (cgate[n][c] + sgate[n][p])          "gated source"
//
//   eds_gated_stats   one read of ONE source at ITS OWN resolution: channel means of the gated values
//                     and the per-pixel dot with this source's slice of w_sse.  Bilinear / nearest x2
//                     upsampling preserves channel means exactly (every low-res pixel carries total
//                     weight 4) and commutes with the dot, so the upsampled source is read at low res.
//   eds_sse_finalize  sgate[n][p] = sigmoid(up2x(dot0)[p] + dot1[p] + b)   (tiny, [N][H][W] scalars)
//   eds_concat_gated  reads the sources again, applies their gates, upsamples source 0, applies the
//                     concat's own gate and writes the conv input ONCE.
//
// Traffic per decoder block: 2 reads of the sources + 1 write of the concat (was 1 read of the sources,
// 2 writes + 1 read of the concat, and 2 reads + 1 write of the block output for attention2).
#include "common.cuh"
#include <cstring>

namespace eds {

constexpr int kGsThreads = 256;
constexpr int kGsUnroll = 8;      // pixels in flight per lane group (memory-level parallelism)

constexpr int ilog2c(int v) { return v <= 1 ? 0 : 1 + ilog2c(v >> 1); }

// Sum d[0..M) over the lanes of a pixel group whose lane-in-group index differs in bit O and below.
// While more than one value is held the exchange is a transpose step (each lane keeps half of the
// values and receives the partner's partial sums of that half), so U values cost about U shuffles
// instead of U * log2(lanes).  Afterwards the lane holds d[0..max(1, U/LPP)) = totals of pixels
// u_sel + q.
template <int O, int M> struct GroupReduce {
    static __device__ __forceinline__ void run(float* d, int l, int& u_sel) {
        if constexpr (O > 0) {
            if constexpr (M > 1) {
                const bool upper = (l & O) != 0;
#pragma unroll
                for (int q = 0; q < M / 2; ++q) {
                    const float send = upper ? d[q] : d[q + M / 2];
                    const float keep = upper ? d[q + M / 2] : d[q];
                    d[q] = keep + __shfl_xor_sync(0xffffffffu, send, O);
                }
                if (upper) u_sel += M / 2;
                GroupReduce<O / 2, M / 2>::run(d, l, u_sel);
            } else {
                d[0] += __shfl_xor_sync(0xffffffffu, d[0], O);
                GroupReduce<O / 2, 1>::run(d, l, u_sel);
            }
        }
    }
};

// ---- pass A -----------------------------------------------------------------------------------
// grid = (pixel chunks, N, 256-channel chunks).  LPP lanes (power of two) share one pixel; lane l
// owns ONE 8-channel vector of every pixel it visits.  With value = v * (cg + s):
//   dot      = sum_c v*(cg*w) + s * sum_c v*w          (two packed FMA chains)
//   chan sum = cg * sum_p v + sum_p s*v                 (accA, accB)
template <typename T, bool GATED, int LPP>
__global__ void __launch_bounds__(kGsThreads, 2)
gated_stats_kernel(const T* __restrict__ x, const float* __restrict__ cgate, const float* __restrict__ sgate, int P,
                   int C, const float* __restrict__ w_sse, float inv_p, float* __restrict__ chan_mean,
                   int mean_stride, int c_off, float* __restrict__ dot, int accumulate) {
    constexpr int PPW = 32 / LPP, U = kGsUnroll;
    constexpr int NS = ilog2c(LPP) < ilog2c(U) ? ilog2c(LPP) : ilog2c(U);   // transpose stages
    constexpr int MF = U >> NS;                                              // totals left per lane
    constexpr int PLAIN = ilog2c(LPP) - NS;                                  // replicated low lane bits
    __shared__ float s_sum[kGsThreads / 32][32][8 + 1];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int l = lane % LPP, sub = lane / LPP;
    const int n = blockIdx.y;
    const int v8 = blockIdx.z * 32 + l;
    const bool live = v8 < C / 8;
    const bool multi = gridDim.z > 1;
    const T* xp = x + (int64_t)n * P * C + (live ? v8 * 8 : 0);
    const float* sg = GATED ? sgate + (int64_t)n * P : nullptr;
    float2 w2[4], cw2[4], cg2[4], accA[4], accB[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) w2[k] = cw2[k] = accA[k] = accB[k] = f2(0.f), cg2[k] = f2(1.f);
    if (live) {
        if (w_sse) ld8f(w_sse + v8 * 8, w2);
        if (GATED) {
            ld8f(cgate + (int64_t)n * C + v8 * 8, cg2);
#pragma unroll
            for (int k = 0; k < 4; ++k) cw2[k] = __fmul2_rn(cg2[k], w2[k]);
        }
    }
    const int per = (P + gridDim.x - 1) / gridDim.x;
    const int p_begin = blockIdx.x * per;
    const int p_end = min(P, p_begin + per);
    constexpr int STEP = (kGsThreads / 32) * PPW * U;
    for (int pb = p_begin + warp * PPW * U; pb < p_end; pb += STEP) {
        float2 v[U][4];
        float sv[U], d[U];
        // All loads are issued unconditionally (addresses clamped into the chunk) so that ptxas
        // keeps U vector loads in flight; lanes without a channel vector read vector 0 and are
        // neutralised by their zero weights, pixels past the end are zeroed in the tail step only.
        const bool tail = pb + PPW * U > p_end;
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int p = min(pb + u * PPW + sub, p_end - 1);
            V8<T>::ld(xp + (int64_t)p * C, v[u]);
            sv[u] = GATED ? __ldg(sg + p) : 0.f;
        }
        if (tail) {
#pragma unroll
            for (int u = 0; u < U; ++u)
                if (pb + u * PPW + sub >= p_end) {
#pragma unroll
                    for (int k = 0; k < 4; ++k) v[u][k] = f2(0.f);
                }
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            float2 a = f2(0.f), b = f2(0.f);
            const float2 s2 = f2(sv[u]);
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                a = __ffma2_rn(v[u][k], w2[k], a);
                accA[k] = __fadd2_rn(accA[k], v[u][k]);
                if (GATED) {
                    b = __ffma2_rn(v[u][k], cw2[k], b);
                    accB[k] = __ffma2_rn(s2, v[u][k], accB[k]);
                }
            }
            d[u] = GATED ? (b.x + b.y) + sv[u] * (a.x + a.y) : (a.x + a.y);
        }
        if (dot) {
            int u_sel = 0;
            GroupReduce<LPP / 2, U>::run(d, l, u_sel);
            if ((l & ((1 << PLAIN) - 1)) == 0) {
#pragma unroll
                for (int q = 0; q < MF; ++q) {
                    const int p = pb + (u_sel + q) * PPW + sub;
                    if (p < p_end) {
                        float* dst = dot + (int64_t)n * P + p;
                        if (multi) atomicAdd(dst, d[q]);
                        else *dst = accumulate ? *dst + d[q] : d[q];
                    }
                }
            }
        }
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const float2 t = GATED ? __ffma2_rn(cg2[k], accA[k], accB[k]) : accA[k];
        s_sum[warp][lane][2 * k] = t.x;
        s_sum[warp][lane][2 * k + 1] = t.y;
    }
    __syncthreads();
    if (threadIdx.x < LPP * 8) {
        const int vl = threadIdx.x >> 3, e = threadIdx.x & 7;
        const int ch = (blockIdx.z * 32 + vl) * 8 + e;
        if (ch < C) {
            float t = 0.f;
            for (int wi = 0; wi < kGsThreads / 32; ++wi)
#pragma unroll
                for (int q = 0; q < PPW; ++q) t += s_sum[wi][q * LPP + vl][e];
            atomicAdd(chan_mean + (int64_t)n * mean_stride + c_off + ch, t * inv_p);
        }
    }
}

// ---- pass A for ALL consumers of a skip source at once ------------------------------------------------------------
// In the dense decoder a block output (or encoder feature) is the same-resolution skip of up to four later blocks,
// each with its own SCSE attention1.  The channel means of the (gated) source do not depend on the consumer and its
// per-pixel dot only differs in the weight slice, so ONE read of the source serves every consumer: K dot maps
// (accumulated into the consumers' dot buffers) and K copies of the channel means (added into the consumers' mean
// rows).  Round 1 read the source once per consumer.  Same lane layout and reductions as gated_stats_kernel; the
// gated value v * (cg + s) is formed once per element and dotted with each consumer's weights.
constexpr int kMaxConsumers = 4;
#ifndef EDS_GS_MULTI_UNROLL
#define EDS_GS_MULTI_UNROLL 8
#endif
constexpr int kGsMultiUnroll = EDS_GS_MULTI_UNROLL;
struct StatConsumers {
    const float* w_sse[kMaxConsumers];    // this source's C-slice of the consumer's sSE weights
    float* chan_mean[kMaxConsumers];      // consumer's [N][mean_stride] rows (+= at c_off)
    float* dot[kMaxConsumers];            // consumer's [N][P] map (+=)
    int mean_stride[kMaxConsumers], c_off[kMaxConsumers];
    int n;
};

template <typename T, bool GATED, int LPP, int K>
__global__ void __launch_bounds__(kGsThreads, 2)
gated_stats_multi_kernel(const T* __restrict__ x, const float* __restrict__ cgate, const float* __restrict__ sgate,
                         int P, int C, float inv_p, StatConsumers cons) {
    constexpr int PPW = 32 / LPP, U = kGsMultiUnroll;                           // pixels in flight per lane group
    constexpr int NS = ilog2c(LPP) < ilog2c(U) ? ilog2c(LPP) : ilog2c(U);
    constexpr int MF = U >> NS;
    constexpr int PLAIN = ilog2c(LPP) - NS;
    __shared__ float s_sum[kGsThreads / 32][32][8 + 1];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int l = lane % LPP, sub = lane / LPP;
    const int n = blockIdx.y;
    const int v8 = blockIdx.z * 32 + l;
    const bool live = v8 < C / 8;
    const T* xp = x + (int64_t)n * P * C + (live ? v8 * 8 : 0);
    const float* sg = GATED ? sgate + (int64_t)n * P : nullptr;
    float2 w2[K][4], cg2[4], acc[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) acc[k] = f2(0.f), cg2[k] = f2(1.f);
#pragma unroll
    for (int c = 0; c < K; ++c)
#pragma unroll
        for (int k = 0; k < 4; ++k) w2[c][k] = f2(0.f);
    if (live) {
#pragma unroll
        for (int c = 0; c < K; ++c) ld8f(cons.w_sse[c] + v8 * 8, w2[c]);
        if (GATED) ld8f(cgate + (int64_t)n * C + v8 * 8, cg2);
    }
    const int per = (P + gridDim.x - 1) / gridDim.x;
    const int p_begin = blockIdx.x * per;
    const int p_end = min(P, p_begin + per);
    constexpr int STEP = (kGsThreads / 32) * PPW * U;
    for (int pb = p_begin + warp * PPW * U; pb < p_end; pb += STEP) {
        float2 v[U][4];
        float sv[U];
        const bool tail = pb + PPW * U > p_end;
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int p = min(pb + u * PPW + sub, p_end - 1);
            V8<T>::ld(xp + (int64_t)p * C, v[u]);
            sv[u] = GATED ? __ldg(sg + p) : 0.f;
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const bool dead = tail && pb + u * PPW + sub >= p_end;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                if (GATED) v[u][k] = __fmul2_rn(v[u][k], __fadd2_rn(cg2[k], f2(sv[u])));
                if (dead || !live) v[u][k] = f2(0.f);
                acc[k] = __fadd2_rn(acc[k], v[u][k]);
            }
        }
#pragma unroll
        for (int c = 0; c < K; ++c) {
            float d[U];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                float2 a = f2(0.f);
#pragma unroll
                for (int k = 0; k < 4; ++k) a = __ffma2_rn(v[u][k], w2[c][k], a);
                d[u] = a.x + a.y;
            }
            int u_sel = 0;
            GroupReduce<LPP / 2, U>::run(d, l, u_sel);
            if ((l & ((1 << PLAIN) - 1)) == 0) {
#pragma unroll
                for (int q = 0; q < MF; ++q) {
                    const int p = pb + (u_sel + q) * PPW + sub;
                    if (p < p_end) {
                        float* dst = cons.dot[c] + (int64_t)n * P + p;
                        if (gridDim.z > 1) atomicAdd(dst, d[q]);
                        else *dst += d[q];
                    }
                }
            }
        }
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        s_sum[warp][lane][2 * k] = acc[k].x;
        s_sum[warp][lane][2 * k + 1] = acc[k].y;
    }
    __syncthreads();
    if (threadIdx.x < LPP * 8) {
        const int vl = threadIdx.x >> 3, e = threadIdx.x & 7;
        const int ch = (blockIdx.z * 32 + vl) * 8 + e;
        if (ch < C) {
            float t = 0.f;
            for (int wi = 0; wi < kGsThreads / 32; ++wi)
#pragma unroll
                for (int q = 0; q < PPW; ++q) t += s_sum[wi][q * LPP + vl][e];
#pragma unroll
            for (int c = 0; c < K; ++c)
                atomicAdd(cons.chan_mean[c] + (int64_t)n * cons.mean_stride[c] + cons.c_off[c] + ch, t * inv_p);
        }
    }
}

// bilinear(align_corners=False) x2 taps of output index o over a source of length len:
// out = (1-l)*src[i0] + l*src[i1]
__device__ __forceinline__ void up2_taps(int o, int len, int& i0, int& i1, float& l) {
    const int i = o >> 1;
    if (o & 1) { i0 = i; i1 = min(i + 1, len - 1); l = 0.25f; }
    else if (i == 0) { i0 = 0; i1 = 0; l = 0.f; }
    else { i0 = i - 1; i1 = i; l = 0.75f; }
}

// sgate[n][p] = sigmoid(up(dot0)[p] + dot1[p] + b) over the OUTPUT grid H x W (= up * h x up * w).
__global__ void __launch_bounds__(256)
sse_finalize_kernel(const float* __restrict__ dot0, const float* __restrict__ dot1, int N, int h, int w, int mode,
                    float b, float* __restrict__ sgate) {
    const int up = mode == EDS_UP_NONE ? 1 : 2;
    const int H = up * h, W = up * w;
    const int64_t total = (int64_t)N * H * W;
    for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
         idx += (int64_t)gridDim.x * blockDim.x) {
        const int ox = (int)(idx % W);
        const int64_t t = idx / W;
        const int oy = (int)(t % H);
        const int n = (int)(t / H);
        float v = b;
        if (dot1) v += dot1[idx];
        if (dot0) {
            const float* d = dot0 + (int64_t)n * h * w;
            if (mode == EDS_UP_NONE) v += d[oy * w + ox];
            else if (mode == EDS_UP_NEAREST) v += d[(oy >> 1) * w + (ox >> 1)];
            else {
                int y0, y1, x0, x1;
                float ly, lx;
                up2_taps(oy, h, y0, y1, ly);
                up2_taps(ox, w, x0, x1, lx);
                const float top = (1.f - lx) * d[y0 * w + x0] + lx * d[y0 * w + x1];
                const float bot = (1.f - lx) * d[y1 * w + x0] + lx * d[y1 * w + x1];
                v += (1.f - ly) * top + ly * bot;
            }
        }
        sgate[idx] = sigmoidf_acc(v);
    }
}

// ---- pass B -----------------------------------------------------------------------------------
struct GatedSrc {
    const void* x;
    const float* cgate;
    const float* sgate;
    int C;
};
struct CatSrcs {
    GatedSrc s[6];
    int n;
};

template <typename T>
__device__ __forceinline__ void ld_gated(const T* p, const float2 (&cg)[4], const float* sg, bool gated,
                                         float2 (&v)[4]) {
    V8<T>::ld(p, v);
    if (gated) {
        const float2 s2 = f2(__ldg(sg));
#pragma unroll
        for (int k = 0; k < 4; ++k) v[k] = __fmul2_rn(v[k], __fadd2_rn(cg[k], s2));
    }
}

// ---- pass A, upsampled part: the channels of source 0 ----------------------------------------------------------------
// One thread = one 8-channel vector of a 2 x 4 OUTPUT block = two adjacent low-res pixels (i, 2jj),
// (i, 2jj+1) of source 0 and their 3 x 4 neighbourhood (12 loads feed 8 outputs; the vertical lerps of
// the two inner columns are shared).  Index arithmetic and bf16 unpacking were most of the instructions
// of the 2 x 2 version; the wider block halves them per output.  grid.x = N*h rows of blocks, grid.y
// covers (jj, vector) of a row; consecutive threads own consecutive vectors of the same block, so every
// global access of a warp is a contiguous run.  All lerps / gates run on the packed fp32 pipe.
template <typename T>
__global__ void __launch_bounds__(256, 2)
concat_gated_kernel(CatSrcs src, int h, int w, int mode, int Ctot, const float* __restrict__ cgate1,
                    const float* __restrict__ sgate1, T* __restrict__ y, int y_stride, int y_coff) {
    const GatedSrc s = src.s[0];
    const uint32_t C8 = (uint32_t)s.C / 8;                              // vectors per pixel of source 0
    const uint32_t wp = (uint32_t)(w + 1) / 2;                          // column pairs per low-res row
    const uint32_t col = blockIdx.y * blockDim.x + threadIdx.x;
    if (col >= wp * C8) return;
    const int jj = (int)(col / C8);
    const int c8 = (int)(col - (uint32_t)jj * C8);
    const int n = (int)(blockIdx.x / (uint32_t)h);
    const int i = (int)(blockIdx.x - (uint32_t)n * h);
    const int j0 = 2 * jj;
    const bool second = j0 + 1 < w;                 // odd widths: the last pair has one column
    const int H = 2 * h, W = 2 * w;
    const int c = c8 * 8;
    const bool gated = s.cgate != nullptr;
    float2 cg[4];
    if (gated) ld8f(s.cgate + (int64_t)n * s.C + c, cg);
    float2 o[8][4];                                 // [row * 4 + column of the block][channel pair]
    const T* xp = reinterpret_cast<const T*>(s.x) + (int64_t)n * h * w * s.C + c;
    const float* sg = s.sgate + (int64_t)n * h * w;      // only dereferenced when gated
    if (mode == EDS_UP_NEAREST) {
        const int p0 = i * w + j0, p1 = i * w + min(j0 + 1, w - 1);
        ld_gated<T>(xp + (int64_t)p0 * s.C, cg, sg + p0, gated, o[0]);
        ld_gated<T>(xp + (int64_t)p1 * s.C, cg, sg + p1, gated, o[2]);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            o[1][q] = o[4][q] = o[5][q] = o[0][q];
            o[3][q] = o[6][q] = o[7][q] = o[2][q];
        }
    } else {
        const int r[3] = {max(i - 1, 0) * w, i * w, min(i + 1, h - 1) * w};
        const int cc[4] = {max(j0 - 1, 0), j0, min(j0 + 1, w - 1), min(j0 + 2, w - 1)};
        float2 top[4][4], bot[4][4];
        const float2 q25 = f2(0.25f), q75 = f2(0.75f);
#pragma unroll
        for (int a = 0; a < 4; ++a) {
            float2 v0[4], v1[4], v2[4];
            ld_gated<T>(xp + (int64_t)(r[0] + cc[a]) * s.C, cg, sg + r[0] + cc[a], gated, v0);
            ld_gated<T>(xp + (int64_t)(r[1] + cc[a]) * s.C, cg, sg + r[1] + cc[a], gated, v1);
            ld_gated<T>(xp + (int64_t)(r[2] + cc[a]) * s.C, cg, sg + r[2] + cc[a], gated, v2);
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const float2 m = __fmul2_rn(q75, v1[q]);
                top[a][q] = __ffma2_rn(q25, v0[q], m);
                bot[a][q] = __ffma2_rn(q25, v2[q], m);
            }
        }
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const float2 t1 = __fmul2_rn(q75, top[1][q]), t2 = __fmul2_rn(q75, top[2][q]);
            const float2 b1 = __fmul2_rn(q75, bot[1][q]), b2 = __fmul2_rn(q75, bot[2][q]);
            o[0][q] = __ffma2_rn(q25, top[0][q], t1);
            o[1][q] = __ffma2_rn(q25, top[2][q], t1);
            o[2][q] = __ffma2_rn(q25, top[1][q], t2);
            o[3][q] = __ffma2_rn(q25, top[3][q], t2);
            o[4][q] = __ffma2_rn(q25, bot[0][q], b1);
            o[5][q] = __ffma2_rn(q25, bot[2][q], b1);
            o[6][q] = __ffma2_rn(q25, bot[1][q], b2);
            o[7][q] = __ffma2_rn(q25, bot[3][q], b2);
        }
    }
    const int64_t p00 = ((int64_t)n * H + 2 * i) * W + 2 * j0;     // output pixel (2i, 2 j0)
    if (cgate1) {
        float2 g1[4];
        ld8f(cgate1 + (int64_t)n * Ctot + c8 * 8, g1);
        float sd[8];
        {
            const float2 a0 = *reinterpret_cast<const float2*>(sgate1 + p00);
            const float2 a1 = *reinterpret_cast<const float2*>(sgate1 + p00 + W);
            sd[0] = a0.x; sd[1] = a0.y; sd[4] = a1.x; sd[5] = a1.y;
            sd[2] = sd[3] = sd[6] = sd[7] = 0.f;
            if (second) {
                const float2 b0 = *reinterpret_cast<const float2*>(sgate1 + p00 + 2);
                const float2 b1 = *reinterpret_cast<const float2*>(sgate1 + p00 + W + 2);
                sd[2] = b0.x; sd[3] = b0.y; sd[6] = b1.x; sd[7] = b1.y;
            }
        }
#pragma unroll
        for (int d = 0; d < 8; ++d) {
            const float2 s1 = f2(sd[d]);
#pragma unroll
            for (int q = 0; q < 4; ++q) o[d][q] = __fmul2_rn(o[d][q], __fadd2_rn(g1[q], s1));
        }
    }
    // y_stride = channels per pixel of the destination map, y_coff = first concat channel it holds
    // (one map of Ctot channels, or one dense map per part so that every pixel row is written whole)
    T* yp = y + p00 * y_stride + (c8 * 8 - y_coff);
    T* yq = yp + (int64_t)W * y_stride;
    V8<T>::st(yp, o[0]);
    V8<T>::st(yp + y_stride, o[1]);
    V8<T>::st(yq, o[4]);
    V8<T>::st(yq + y_stride, o[5]);
    if (second) {
        V8<T>::st(yp + 2 * y_stride, o[2]);
        V8<T>::st(yp + 3 * y_stride, o[3]);
        V8<T>::st(yq + 2 * y_stride, o[6]);
        V8<T>::st(yq + 3 * y_stride, o[7]);
    }
}

// ---- pass B, same-resolution (skip) part: a lean streaming kernel ---------------------------------------------------
// One thread = one 8-channel vector of FOUR consecutive pixels of a row.  (A version that kept eight output vectors
// per thread, the 2 x 4 block of pass A, needed 128 registers, spilled in the bf16 build and was latency-bound at
// 23 % occupancy.)  grid.x = N * H rows, grid.y covers (quad, vector) of a row.
template <typename T>
__global__ void __launch_bounds__(256, 3)
concat_skip_kernel(CatSrcs src, int H, int W, int Ctot, const float* __restrict__ cgate1,
                   const float* __restrict__ sgate1, T* __restrict__ y, int y_stride, int y_coff) {
    const uint32_t C8a = (uint32_t)src.s[0].C / 8;
    const uint32_t C8 = (uint32_t)Ctot / 8 - C8a;                  // vectors per pixel of the skip part
    const uint32_t quads = (uint32_t)(W + 3) / 4;
    const uint32_t col = blockIdx.y * blockDim.x + threadIdx.x;
    if (col >= quads * C8) return;
    const int qx = (int)(col / C8);
    const int c8 = (int)(col - (uint32_t)qx * C8) + (int)C8a;      // vector inside the concat
    const int n = (int)(blockIdx.x / (uint32_t)H);
    const int yy = (int)(blockIdx.x - (uint32_t)n * H);
    const int x0 = 4 * qx;
    const int npx = min(4, W - x0);
    int c = c8 * 8, k = 0;
    while (k < src.n - 1 && c >= src.s[k].C) { c -= src.s[k].C; ++k; }
    const GatedSrc sk = src.s[k];
    const bool gated = sk.cgate != nullptr;
    float2 cg[4];
    if (gated) ld8f(sk.cgate + (int64_t)n * sk.C + c, cg);
    const int64_t p0 = ((int64_t)n * H + yy) * W + x0;             // first pixel of the quad
    const T* xp = reinterpret_cast<const T*>(sk.x) + p0 * sk.C + c;
    const float* sg = sk.sgate + p0;                               // only dereferenced when gated
    float2 o[4][4];
#pragma unroll
    for (int d = 0; d < 4; ++d) {
        const int dd = min(d, npx - 1);                            // clamped address for a ragged last quad
        ld_gated<T>(xp + (int64_t)dd * sk.C, cg, sg + dd, gated, o[d]);
    }
    if (cgate1) {
        float2 g1[4];
        ld8f(cgate1 + (int64_t)n * Ctot + c8 * 8, g1);
#pragma unroll
        for (int d = 0; d < 4; ++d) {
            const float2 s1 = f2(__ldg(sgate1 + p0 + min(d, npx - 1)));
#pragma unroll
            for (int q = 0; q < 4; ++q) o[d][q] = __fmul2_rn(o[d][q], __fadd2_rn(g1[q], s1));
        }
    }
    T* yp = y + p0 * y_stride + (c8 * 8 - y_coff);
#pragma unroll
    for (int d = 0; d < 4; ++d)
        if (d < npx) V8<T>::st(yp + (int64_t)d * y_stride, o[d]);
}

// y = x * (cgate[n][c] + sgate[n][p]) for an already materialised map (gate = probabilities).
template <typename T>
__global__ void __launch_bounds__(256)
apply_gate_kernel(const T* __restrict__ x, const float* __restrict__ cgate, const float* __restrict__ sgate, int HW,
                  int C8, int64_t total, T* __restrict__ y) {
    for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
         idx += (int64_t)gridDim.x * blockDim.x) {
        const int64_t pix = idx / C8;
        const int c8 = (int)(idx - pix * C8);
        const int n = (int)(pix / HW);
        const float s = __ldg(sgate + pix);
        const float4* g4 = reinterpret_cast<const float4*>(cgate + (int64_t)n * C8 * 8 + c8 * 8);
        const float4 g0 = __ldg(g4), g1 = __ldg(g4 + 1);
        const float g[8] = {g0.x, g0.y, g0.z, g0.w, g1.x, g1.y, g1.z, g1.w};
        float v[8];
        Vec8<T>::ld(x + idx * 8, v);
#pragma unroll
        for (int i = 0; i < 8; ++i) v[i] *= g[i] + s;
        Vec8<T>::st(y + idx * 8, v);
    }
}

}  // namespace eds

using namespace eds;

extern "C" int eds_gated_stats(const void* x, const float* cgate, const float* sgate, int N, int P, int C,
                               const float* w_sse, float* chan_mean, int mean_stride, int c_off, int zero_mean,
                               float* dot, int accumulate, int dtype, void* stream) {
    EDS_REQUIRE(x && chan_mean, "gated_stats: null pointer");
    EDS_REQUIRE((cgate == nullptr) == (sgate == nullptr), "gated_stats: cgate and sgate come together");
    EDS_REQUIRE(N > 0 && N <= 65535 && P > 0 && C > 0 && C % 8 == 0, "gated_stats: bad shape N=%d P=%d C=%d", N, P, C);
    EDS_REQUIRE(mean_stride >= c_off + C && c_off >= 0 && c_off % 8 == 0, "gated_stats: bad mean layout");
    EDS_REQUIRE(!dot || w_sse, "gated_stats: dot requested without w_sse");
    const int c8 = C / 8;
    int lpp = 32;
    while (lpp > 1 && lpp / 2 >= c8) lpp /= 2;
    const int zchunks = ceil_div(c8, 32);
    EDS_REQUIRE(zchunks <= 65535, "gated_stats: too many channels");
    cudaError_t e = cudaSuccess;
    if (zero_mean) e = cudaMemsetAsync(chan_mean, 0, sizeof(float) * (size_t)N * mean_stride, as_stream(stream));
    if (e == cudaSuccess && dot && zchunks > 1 && !accumulate)
        e = cudaMemsetAsync(dot, 0, sizeof(float) * (size_t)N * P, as_stream(stream));
    if (e != cudaSuccess) {
        set_error("gated_stats: memset failed: %s", cudaGetErrorString(e));
        return EDS_ERR_CUDA;
    }
    int chunks = ceil_div(148 * 12, N * zchunks);
    const int max_chunks = ceil_div(P, 8 * (32 / lpp) * kGsUnroll);
    if (chunks > max_chunks) chunks = max_chunks;
    if (chunks < 1) chunks = 1;
    dim3 grid(chunks, N, zchunks);
#define EDS_GS_LAUNCH(T, G, L)                                                                                   \
    gated_stats_kernel<T, G, L><<<grid, kGsThreads, 0, as_stream(stream)>>>(                                     \
        (const T*)x, cgate, sgate, P, C, w_sse, 1.0f / (float)P, chan_mean, mean_stride, c_off, dot, accumulate)
#define EDS_GS_LPP(T, G)                                                                                         \
    switch (lpp) {                                                                                               \
        case 1: EDS_GS_LAUNCH(T, G, 1); break;                                                                   \
        case 2: EDS_GS_LAUNCH(T, G, 2); break;                                                                   \
        case 4: EDS_GS_LAUNCH(T, G, 4); break;                                                                   \
        case 8: EDS_GS_LAUNCH(T, G, 8); break;                                                                   \
        case 16: EDS_GS_LAUNCH(T, G, 16); break;                                                                 \
        default: EDS_GS_LAUNCH(T, G, 32); break;                                                                 \
    }
    EDS_DISPATCH_DTYPE(dtype, T, {
        if (cgate) { EDS_GS_LPP(T, true) } else { EDS_GS_LPP(T, false) }
    });
#undef EDS_GS_LPP
#undef EDS_GS_LAUNCH
    return check_launch("gated_stats_kernel");
}

template <typename T, bool GATED, int LPP>
static void stats_multi_launch(int K, dim3 grid, cudaStream_t st, const void* x, const float* cgate, const float* sgate,
                               int P, int C, const StatConsumers& cons) {
    const float inv_p = 1.0f / (float)P;
    switch (K) {
        case 1: gated_stats_multi_kernel<T, GATED, LPP, 1><<<grid, kGsThreads, 0, st>>>((const T*)x, cgate, sgate, P, C, inv_p, cons); break;
        case 2: gated_stats_multi_kernel<T, GATED, LPP, 2><<<grid, kGsThreads, 0, st>>>((const T*)x, cgate, sgate, P, C, inv_p, cons); break;
        case 3: gated_stats_multi_kernel<T, GATED, LPP, 3><<<grid, kGsThreads, 0, st>>>((const T*)x, cgate, sgate, P, C, inv_p, cons); break;
        default: gated_stats_multi_kernel<T, GATED, LPP, 4><<<grid, kGsThreads, 0, st>>>((const T*)x, cgate, sgate, P, C, inv_p, cons); break;
    }
}

extern "C" int eds_gated_stats_multi(const void* x, const float* cgate, const float* sgate, int N, int P, int C,
                                     int n_consumers, const float* const* w_sse, float* const* chan_mean,
                                     const int* mean_stride, const int* c_off, float* const* dot, int dtype,
                                     void* stream) {
    EDS_REQUIRE(x && w_sse && chan_mean && mean_stride && c_off && dot, "gated_stats_multi: null pointer");
    EDS_REQUIRE((cgate == nullptr) == (sgate == nullptr), "gated_stats_multi: cgate and sgate come together");
    EDS_REQUIRE(N > 0 && N <= 65535 && P > 0 && C > 0 && C % 8 == 0, "gated_stats_multi: bad shape N=%d P=%d C=%d", N, P, C);
    EDS_REQUIRE(n_consumers >= 1 && n_consumers <= kMaxConsumers, "gated_stats_multi: n_consumers=%d (1..%d)",
                n_consumers, kMaxConsumers);
    StatConsumers cons;
    memset(&cons, 0, sizeof(cons));
    cons.n = n_consumers;
    for (int k = 0; k < n_consumers; ++k) {
        EDS_REQUIRE(w_sse[k] && chan_mean[k] && dot[k], "gated_stats_multi: consumer %d: null pointer", k);
        EDS_REQUIRE(mean_stride[k] >= c_off[k] + C && c_off[k] >= 0 && c_off[k] % 8 == 0,
                    "gated_stats_multi: consumer %d: bad mean layout", k);
        cons.w_sse[k] = w_sse[k]; cons.chan_mean[k] = chan_mean[k]; cons.dot[k] = dot[k];
        cons.mean_stride[k] = mean_stride[k]; cons.c_off[k] = c_off[k];
    }
    const int c8 = C / 8;
    int lpp = 32;
    while (lpp > 1 && lpp / 2 >= c8) lpp /= 2;
    const int zchunks = ceil_div(c8, 32);
    EDS_REQUIRE(zchunks <= 65535, "gated_stats_multi: too many channels");
    int chunks = ceil_div(148 * 12, N * zchunks);
    const int max_chunks = ceil_div(P, 8 * (32 / lpp) * kGsMultiUnroll);
    if (chunks > max_chunks) chunks = max_chunks;
    if (chunks < 1) chunks = 1;
    dim3 grid(chunks, N, zchunks);
    cudaStream_t st = as_stream(stream);
#define EDS_GSM_LPP(T, G)                                                                                        \
    switch (lpp) {                                                                                               \
        case 1: stats_multi_launch<T, G, 1>(n_consumers, grid, st, x, cgate, sgate, P, C, cons); break;          \
        case 2: stats_multi_launch<T, G, 2>(n_consumers, grid, st, x, cgate, sgate, P, C, cons); break;          \
        case 4: stats_multi_launch<T, G, 4>(n_consumers, grid, st, x, cgate, sgate, P, C, cons); break;          \
        case 8: stats_multi_launch<T, G, 8>(n_consumers, grid, st, x, cgate, sgate, P, C, cons); break;          \
        case 16: stats_multi_launch<T, G, 16>(n_consumers, grid, st, x, cgate, sgate, P, C, cons); break;        \
        default: stats_multi_launch<T, G, 32>(n_consumers, grid, st, x, cgate, sgate, P, C, cons); break;        \
    }
    EDS_DISPATCH_DTYPE(dtype, T, {
        if (cgate) { EDS_GSM_LPP(T, true) } else { EDS_GSM_LPP(T, false) }
    });
#undef EDS_GSM_LPP
    return check_launch("gated_stats_multi_kernel");
}

extern "C" int eds_sse_finalize(const float* dot0, const float* dot1, int N, int h, int w, int mode, float b_sse,
                                float* sgate, void* stream) {
    EDS_REQUIRE(sgate && (dot0 || dot1), "sse_finalize: null pointer");
    EDS_REQUIRE(mode == EDS_UP_NEAREST || mode == EDS_UP_BILINEAR || mode == EDS_UP_NONE, "sse_finalize: bad mode %d",
                mode);
    EDS_REQUIRE(N > 0 && h > 0 && w > 0, "sse_finalize: bad shape");
    const int up = mode == EDS_UP_NONE ? 1 : 2;
    const int64_t total = (int64_t)N * up * h * up * w;
    int64_t blocks = (total + 255) / 256;
    if (blocks > 148 * 8) blocks = 148 * 8;
    sse_finalize_kernel<<<(unsigned)blocks, 256, 0, as_stream(stream)>>>(dot0, dot1, N, h, w, mode, b_sse, sgate);
    return check_launch("sse_finalize_kernel");
}

static int concat_gated_launch(const eds_gated_src* srcs, int n_srcs, int N, int h, int w, int mode,
                               const float* cgate, const float* sgate, void* y, void* y_skip, int dtype,
                               void* stream) {
    EDS_REQUIRE(srcs && y, "concat_gated: null pointer");
    EDS_REQUIRE(n_srcs >= 1 && n_srcs <= 6, "concat_gated: n_srcs=%d not in 1..6", n_srcs);
    EDS_REQUIRE(mode == EDS_UP_NEAREST || mode == EDS_UP_BILINEAR, "concat_gated: mode %d (nearest / bilinear x2 only)",
                mode);
    EDS_REQUIRE((cgate == nullptr) == (sgate == nullptr), "concat_gated: cgate and sgate come together");
    EDS_REQUIRE(N > 0 && h > 0 && w > 0, "concat_gated: bad shape");
    CatSrcs cs;
    cs.n = n_srcs;
    int Ctot = 0;
    for (int k = 0; k < 6; ++k) {
        if (k < n_srcs) {
            EDS_REQUIRE(srcs[k].x && srcs[k].C > 0 && srcs[k].C % 8 == 0, "concat_gated: bad source %d", k);
            EDS_REQUIRE((srcs[k].cgate == nullptr) == (srcs[k].sgate == nullptr),
                        "concat_gated: source %d: cgate and sgate come together", k);
            cs.s[k].x = srcs[k].x; cs.s[k].cgate = srcs[k].cgate; cs.s[k].sgate = srcs[k].sgate; cs.s[k].C = srcs[k].C;
            Ctot += srcs[k].C;
        } else {
            cs.s[k].x = nullptr; cs.s[k].cgate = nullptr; cs.s[k].sgate = nullptr; cs.s[k].C = 0;
        }
    }
    const int c8a = cs.s[0].C / 8, c8b = Ctot / 8 - c8a;
    EDS_REQUIRE((int64_t)w * (Ctot / 8) < (1ll << 24) && (int64_t)N * h < (1ll << 31), "concat_gated: map too large");
    EDS_REQUIRE(c8b == 0 || (int64_t)N * 2 * h < (1ll << 31), "concat_gated: map too large (N * 2h = %lld rows)",
                (long long)N * 2 * h);
    const int wp = (w + 1) / 2;
    EDS_REQUIRE(!y_skip || c8b > 0, "concat_gated: y_skip given without skip sources");
    // one destination of Ctot channels, or two dense ones (upsampled part / skip part)
    const int stride_a = y_skip ? cs.s[0].C : Ctot;
    // (A shared-memory tiled variant of this part -- neighbourhood gated once per CTA, fp32 tile, 2 x 4 output blocks
    // per thread -- measured 2.4-2.5 TB/s against 3.3-3.7 TB/s for the per-thread kernel on the benchmark's layers,
    // scripts/dev_concat_probe.py: one barrier per small tile and 104 registers leave too little in flight.)
    dim3 grid_a((unsigned)(N * h), (unsigned)ceil_div(wp * c8a, 256));
    EDS_DISPATCH_DTYPE(dtype, T, (concat_gated_kernel<T><<<grid_a, 256, 0, as_stream(stream)>>>(
                                     cs, h, w, mode, Ctot, cgate, sgate, (T*)y, stride_a, 0)));
    if (c8b > 0) {
        void* yb = y_skip ? y_skip : y;
        const int stride_b = y_skip ? Ctot - cs.s[0].C : Ctot;
        const int coff_b = y_skip ? cs.s[0].C : 0;
        dim3 grid_s((unsigned)(N * 2 * h), (unsigned)ceil_div(ceil_div(2 * w, 4) * c8b, 256));
        EDS_DISPATCH_DTYPE(dtype, T, (concat_skip_kernel<T><<<grid_s, 256, 0, as_stream(stream)>>>(
                                         cs, 2 * h, 2 * w, Ctot, cgate, sgate, (T*)yb, stride_b, coff_b)));
    }
    return check_launch("concat_gated_kernel");
}

extern "C" int eds_concat_gated(const eds_gated_src* srcs, int n_srcs, int N, int h, int w, int mode,
                                const float* cgate, const float* sgate, void* y, int dtype, void* stream) {
    return concat_gated_launch(srcs, n_srcs, N, h, w, mode, cgate, sgate, y, nullptr, dtype, stream);
}

extern "C" int eds_concat_gated_split(const eds_gated_src* srcs, int n_srcs, int N, int h, int w, int mode,
                                      const float* cgate, const float* sgate, void* y_up, void* y_skip, int dtype,
                                      void* stream) {
    EDS_REQUIRE(y_skip, "concat_gated_split: null pointer");
    return concat_gated_launch(srcs, n_srcs, N, h, w, mode, cgate, sgate, y_up, y_skip, dtype, stream);
}

extern "C" int eds_apply_gate(const void* x, const float* cgate, const float* sgate, int N, int HW, int C, void* y,
                              int dtype, void* stream) {
    EDS_REQUIRE(x && cgate && sgate && y, "apply_gate: null pointer");
    EDS_REQUIRE(C % 8 == 0 && C > 0 && N > 0 && HW > 0, "apply_gate: bad shape");
    const int64_t total = (int64_t)N * HW * (C / 8);
    int64_t blocks = (total + 255) / 256;
    if (blocks > 148 * 16) blocks = 148 * 16;
    EDS_DISPATCH_DTYPE(dtype, T, (apply_gate_kernel<T><<<(unsigned)blocks, 256, 0, as_stream(stream)>>>(
                                     (const T*)x, cgate, sgate, HW, C / 8, total, (T*)y)));
    return check_launch("apply_gate_kernel");
}
