// TTA de-augment + mean + sigmoid, bilinear paste, and sliding-window tile fetch.
//
// Replaces (reference file:line):
//   - ttach.SegmentationTTAWrapper de-augmentation and Merger('mean') as used at
//     src/main/tta.py:92-99,173-180, followed by the sigmoid of tta.py:114,210;
//   - cv2.resize(..., INTER_LINEAR) + `preds[x1:x2, y1:y2] = tile` (tta.py:211-213)
//     and center_crop + GF.resize (tta.py:117-119);
//   - dataset.read(window) + A.Resize + preprocessing_fn + ToTensorV2 (tta.py:201-204).
// All are HBM-bound streaming kernels; the flip / rot90 views are never materialised, they are index maps applied
// while reading.  tta_blend_x2_kernel does merge + sigmoid + x2 + overwrite-paste in one pass (the product path for
// tile sizes that are multiples of 64); tta_merge*_kernel / paste_tiles_x2_kernel / resize_paste_kernel are the
// pieces (generic TTA wrapper, ensemble mean, whole-image path, other tile sizes); the Gaussian kernels are an
// opt-in blend mode with no reference counterpart.
#include "common.cuh"

namespace eds {

struct ViewMaps {
    int m[8][6];
};

// One CTA (32 x 8 threads) = one 32x32 output tile of one image; a thread owns 4 rows of its column.
// All 4 x V loads of a thread are issued before the first use (addresses clamped into the tile, so no
// load is conditional) -- 32 x 4 B in flight per thread; views whose map transposes the axes are read
// along THEIR rows (coalesced) and turned through one shared-memory tile per view.  The sum runs in
// view order in fp32, like ttach's Merger.
__global__ void __launch_bounds__(256)
tta_merge_kernel(const float* __restrict__ logits, int V, int B, int S, ViewMaps maps, int apply_sigmoid,
                 float* __restrict__ prob) {
    __shared__ float tile[8][32][33];
    const int tx = threadIdx.x, ty = threadIdx.y;       // 32 x 8
    const int b = blockIdx.z;
    const int j = blockIdx.x * 32 + tx;                 // output col
    const int jc = min(j, S - 1);
    float val[4][8];
    bool any_t = false;
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        const int rr = ty + 8 * r;                       // row inside the tile
        const int ic = min(blockIdx.y * 32 + rr, S - 1);
        // transposing views: thread (rr,tx) fetches the value of output (row tx, col rr) of the tile
        const int io = min(blockIdx.y * 32 + tx, S - 1), jo = min(blockIdx.x * 32 + rr, S - 1);
#pragma unroll
        for (int v = 0; v < 8; ++v) {
            val[r][v] = 0.f;
            if (v < V) {
                const int* m = maps.m[v];
                const float* src = logits + ((int64_t)v * B + b) * S * S;
                if (m[1] == 0) {
                    val[r][v] = __ldg(src + (int64_t)(m[0] * ic + m[2]) * S + (m[4] * jc + m[5]));
                } else {
                    val[r][v] = __ldg(src + (int64_t)(m[1] * jo + m[2]) * S + (m[3] * io + m[5]));
                    any_t = true;
                }
            }
        }
    }
    if (any_t) {                       // CTA-uniform (the maps are kernel parameters)
#pragma unroll
        for (int r = 0; r < 4; ++r)
#pragma unroll
            for (int v = 0; v < 8; ++v)
                if (v < V && maps.m[v][1] != 0) tile[v][tx][ty + 8 * r] = val[r][v];
        __syncthreads();
#pragma unroll
        for (int r = 0; r < 4; ++r)
#pragma unroll
            for (int v = 0; v < 8; ++v)
                if (v < V && maps.m[v][1] != 0) val[r][v] = tile[v][ty + 8 * r][tx];
    }
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        const int i = blockIdx.y * 32 + ty + 8 * r;
        float acc = val[r][0];
#pragma unroll
        for (int v = 1; v < 8; ++v)
            if (v < V) acc += val[r][v];
        if (i < S && j < S) {
            const float mean = acc / (float)V;
            prob[((int64_t)b * S + i) * S + j] = apply_sigmoid ? sigmoidf_acc(mean) : mean;
        }
    }
}

// The same merge for S % 64 == 0 (every production tile size): one CTA (1024 / ROWS threads) = one 64x64 output
// tile, a thread owns ROWS rows x 4 adjacent columns and moves 16-byte vectors only -- a quarter of the load
// instructions of the kernel above and no per-element address arithmetic, which is what bounded it
// (issue-bound at 0.40 of HBM peak).  Views are taken in two groups of four (4 * ROWS vector loads in flight per
// thread, two CTAs per SM); the running sum is still formed in view order, so the result is bit-identical.
// Transposing views are read along THEIR rows and turned through shared memory: [64][64] floats per view,
// column index XORed with f(row) = ((row>>2)&7)<<2 | ((row>>5)&1)<<1, which makes the scalar stores of a
// warp hit 32 distinct banks and keeps every aligned group of 4 columns inside one 16-byte word (its two
// pairs swapped when bit 5 of the row is set) so the read-back is one LDS.128.
constexpr int kMergeTile = 64;
__device__ __forceinline__ int merge_swz(int row) { return (((row >> 2) & 7) << 2) | (((row >> 5) & 1) << 1); }

template <int ROWS, int MINB>
__global__ void __launch_bounds__(1024 / ROWS, MINB)
tta_merge64_kernel(const float* __restrict__ logits, int V, int B, int S, ViewMaps maps, int apply_sigmoid,
                   float* __restrict__ prob) {
    extern __shared__ __align__(16) float mtile[];      // [4][64][64]
    const int tid = threadIdx.x;
    const int l16 = tid & 15, rg = tid >> 4;
    const int b = blockIdx.z;
    const int I0 = blockIdx.y * kMergeTile, J0 = blockIdx.x * kMergeTile;
    constexpr int RSTEP = kMergeTile / ROWS;   // rows rg + RSTEP * r
    float4 acc[ROWS];
#pragma unroll
    for (int g = 0; g < 2; ++g) {
        if (g * 4 >= V) break;
        float4 val[4][ROWS];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int v = g * 4 + u;
            if (v >= V) continue;
            const int* m = maps.m[v];
            const float* src = logits + ((int64_t)v * B + b) * S * S;
            if (m[1] == 0) {       // straight: output (i, j..j+3) <- source row m0*i+m2, columns m4*j+m5 (reversed if m4<0)
                const float* p = src + (m[4] > 0 ? J0 + 4 * l16 + m[5] : m[5] - J0 - 4 * l16 - 3);
#pragma unroll
                for (int r = 0; r < ROWS; ++r)
                    val[u][r] = __ldg(reinterpret_cast<const float4*>(p + (int64_t)(m[0] * (I0 + rg + RSTEP * r) + m[2]) * S));
            } else {               // transposing: the tile's source block, rows q = rg + 16r, columns 4*l16..+3
                const int row0 = m[1] > 0 ? J0 + m[2] : m[2] - J0 - (kMergeTile - 1);
                const int col0 = m[3] > 0 ? I0 + m[5] : m[5] - I0 - (kMergeTile - 1);
                const float* p = src + (int64_t)(row0 + rg) * S + col0 + 4 * l16;
#pragma unroll
                for (int r = 0; r < ROWS; ++r)
                    val[u][r] = __ldg(reinterpret_cast<const float4*>(p + (int64_t)(RSTEP * r) * S));
            }
        }
        if (g) __syncthreads();        // the previous group's tiles have been read
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int v = g * 4 + u;
            if (v >= V || maps.m[v][1] == 0) continue;
            const int* m = maps.m[v];
            float* t = mtile + u * kMergeTile * kMergeTile;
#pragma unroll
            for (int r = 0; r < ROWS; ++r) {
                const int q = rg + RSTEP * r;
                const int jl = m[1] > 0 ? q : kMergeTile - 1 - q;
                const float e[4] = {val[u][r].x, val[u][r].y, val[u][r].z, val[u][r].w};
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const int il = m[3] > 0 ? 4 * l16 + k : kMergeTile - 1 - 4 * l16 - k;
                    t[il * kMergeTile + (jl ^ merge_swz(il))] = e[k];
                }
            }
        }
        __syncthreads();
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int v = g * 4 + u;
            if (v >= V) continue;
            const int* m = maps.m[v];
#pragma unroll
            for (int r = 0; r < ROWS; ++r) {
                float4 x = val[u][r];
                if (m[1] == 0) {
                    if (m[4] < 0) x = make_float4(x.w, x.z, x.y, x.x);
                } else {
                    const int il = rg + RSTEP * r;
                    const float4 w = *reinterpret_cast<const float4*>(mtile + u * kMergeTile * kMergeTile +
                                                                      il * kMergeTile + ((l16 ^ ((il >> 2) & 7)) << 2));
                    x = (il & 32) ? make_float4(w.z, w.w, w.x, w.y) : w;
                }
                if (v == 0) acc[r] = x;
                else { acc[r].x += x.x; acc[r].y += x.y; acc[r].z += x.z; acc[r].w += x.w; }
            }
        }
    }
    const float fv = (float)V;
#pragma unroll
    for (int r = 0; r < ROWS; ++r) {
        float4 o = make_float4(acc[r].x / fv, acc[r].y / fv, acc[r].z / fv, acc[r].w / fv);
        if (apply_sigmoid) o = make_float4(sigmoidf_acc(o.x), sigmoidf_acc(o.y), sigmoidf_acc(o.z), sigmoidf_acc(o.w));
        *reinterpret_cast<float4*>(prob + ((int64_t)b * S + I0 + rg + RSTEP * r) * S + J0 + 4 * l16) = o;
    }
}

// Bilinear resize + overwrite paste.  Coordinate arithmetic follows cv2's resizeLinear for CV_32F
// (double coordinates, float weights, horizontal pass then vertical pass).  A CTA covers a 64 x 32
// block of the output; its 64 column and 32 row coordinates are computed ONCE in double precision
// (fp64 is a trickle pipe on this chip) into shared memory, then every thread produces 8 pixels.
constexpr int kPasteBX = 64, kPasteBY = 32;
__global__ void __launch_bounds__(256)
resize_paste_kernel(const float* __restrict__ src, int src_w, int crop_y, int crop_x, int crop_h,
                    int crop_w, float* __restrict__ dst, int dst_h, int dst_w, int dst_y,
                    int dst_x, int out_h, int out_w, double scale_y, double scale_x) {
    __shared__ int s_i0[kPasteBX + kPasteBY], s_i1[kPasteBX + kPasteBY];
    __shared__ float s_f[kPasteBX + kPasteBY];
    const int tid = threadIdx.y * blockDim.x + threadIdx.x;
    const int bx0 = blockIdx.x * kPasteBX, by0 = blockIdx.y * kPasteBY;
    if (tid < kPasteBX + kPasteBY) {
        // source coordinate in double, fraction rounded to float once (matches cv2 4.x to 2e-7;
        // rounding the coordinate itself to float would cost 5e-5 at x ~ 1000)
        const bool is_x = tid < kPasteBX;
        const int o = is_x ? bx0 + tid : by0 + (tid - kPasteBX);
        const int lim = is_x ? crop_w : crop_h;
        const double d = (o + 0.5) * (is_x ? scale_x : scale_y) - 0.5;
        int s0 = (int)floor(d);
        float f = (float)(d - (double)s0);
        if (s0 < 0) { s0 = 0; f = 0.f; }
        if (s0 >= lim - 1) { s0 = lim - 1; f = 0.f; }
        s_i0[tid] = s0;
        s_i1[tid] = s0 + 1 < lim ? s0 + 1 : lim - 1;
        s_f[tid] = f;
    }
    __syncthreads();
    const int lx = tid & 63;                 // column inside the block
    const int ox = bx0 + lx;
    const int gx = dst_x + ox;
    if (ox >= out_w || gx < 0 || gx >= dst_w) return;
    const int sx = s_i0[lx], sx1 = s_i1[lx];
    const float a1 = s_f[lx], a0 = 1.f - a1;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        const int ly = (tid >> 6) + 4 * k;   // 4 rows per pass, 8 passes
        const int oy = by0 + ly;
        const int gy = dst_y + oy;
        if (oy >= out_h || gy < 0 || gy >= dst_h) continue;
        const int sy = s_i0[kPasteBX + ly], sy1 = s_i1[kPasteBX + ly];
        const float b1 = s_f[kPasteBX + ly], b0 = 1.f - b1;
        const float* r0 = src + (int64_t)(crop_y + sy) * src_w + crop_x;
        const float* r1 = src + (int64_t)(crop_y + sy1) * src_w + crop_x;
        const float h0 = __fadd_rn(__fmul_rn(__ldg(r0 + sx), a0), __fmul_rn(__ldg(r0 + sx1), a1));
        const float h1 = __fadd_rn(__fmul_rn(__ldg(r1 + sx), a0), __fmul_rn(__ldg(r1 + sx1), a1));
        dst[(int64_t)gy * dst_w + gx] = __fadd_rn(__fmul_rn(h0, b0), __fmul_rn(h1, b1));
    }
}

// All tiles of a batch in ONE launch: dst[ys[b] + oy][xs[b] + ox] = bilinear x2 of src[b] (S x S -> 2S x 2S),
// tiles pasted in index order with last-writer-wins (tta.py:211-213: `preds[x1:x2, y1:y2] = tile` in make_grid
// order).  Concurrent CTAs must not race on the overlaps, so a pixel of tile b is written only if no later
// tile of the batch covers it -- the same final image, fewer bytes written.  Arithmetic is resize_paste's for
// the exact scale 1/2 (fractions 0 / 0.25 / 0.75, horizontal pass then vertical pass, unfused mul + add),
// so the two kernels agree bit for bit.
constexpr int kPasteMaxTiles = 32;
struct PasteTiles {
    int y[kPasteMaxTiles], x[kPasteMaxTiles];
    int n;
};

// One thread = 4 output columns that are 16-byte ALIGNED IN dst (tile origins are arbitrary, e.g. x = 1429) x
// kPasteRows output rows: kPasteRows/2 + 2 source rows x 3-4 source columns are read (round 1: 12 scalar loads and 8
// scalar stores per 8 pixels, issue-bound at 1.25 TB/s), the results leave as 128-bit stores.  Blocks that a
// later tile covers completely return before their first load (with make_grid's overlaps that is half of all blocks).
// grid = (ceil((2S + 3) / 256), ceil(2S / (4 * kPasteRows)), tiles in src), block = (64, 4).
constexpr int kPasteRows = 16;
__global__ void __launch_bounds__(256)
paste_tiles_x2_kernel(const float* __restrict__ src, int S, PasteTiles tiles, int first_tile, float* __restrict__ dst,
                      int dst_h, int dst_w) {
    const int b = first_tile + blockIdx.z;              // index into the tile list; src holds tiles first_tile ..
    const float* sp = src + (int64_t)blockIdx.z * S * S;
    const int ty0 = tiles.y[b], tx0 = tiles.x[b];
    const int out = 2 * S;
    const int tid = threadIdx.y * blockDim.x + threadIdx.x;
    // aligned quads of dst columns covering [tx0, tx0 + out): quad index q -> columns gq .. gq+3
    const int gq = (tx0 & ~3) + 4 * (blockIdx.x * 64 + (tid & 63));
    if (gq >= tx0 + out || gq + 3 < tx0 || gq >= dst_w) return;
    const int a = (blockIdx.y * (4 * kPasteRows) + (tid >> 6) * kPasteRows) >> 1;      // output rows 2a .. 2a+kPasteRows-1
    const int gy_lo = ty0 + 2 * a, gy_hi = gy_lo + kPasteRows - 1;
    if (gy_lo >= dst_h || gy_hi < 0 || 2 * a >= out) return;
    // later tiles (last writer wins): fully covered -> nothing to do; partly covered -> per-pixel test below
    unsigned later = 0;
    for (int l = b + 1; l < tiles.n; ++l) {
        const int lx = tiles.x[l], ly = tiles.y[l];
        const bool cols_all = gq >= lx && gq + 3 < lx + out, cols_any = gq + 3 >= lx && gq < lx + out;
        const bool rows_all = gy_lo >= ly && gy_hi < ly + out, rows_any = gy_hi >= ly && gy_lo < ly + out;
        if (cols_all && rows_all) return;
        if (cols_any && rows_any) later |= 1u << l;
    }
    // horizontal pass: output column ox of the tile blends source columns sx, sx+1 with weights (1-a1, a1)
    int sx[4], sx1[4];
    float a0[4], a1[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const int ox = min(max(gq + j - tx0, 0), out - 1);           // columns outside the tile are never stored
        int c = (ox >> 1) - ((ox & 1) ? 0 : 1);
        float f = (ox & 1) ? 0.25f : 0.75f;
        if (c < 0) { c = 0; f = 0.f; }
        if (c >= S - 1) { c = S - 1; f = 0.f; }
        sx[j] = c;
        sx1[j] = min(c + 1, S - 1);
        a1[j] = f;
        a0[j] = 1.f - f;
    }
    constexpr int kSrcRows = kPasteRows / 2 + 2;
    float h[kSrcRows][4];
#pragma unroll
    for (int t = 0; t < kSrcRows; ++t) {
        const float* row = sp + (int64_t)min(max(a - 1 + t, 0), S - 1) * S;
#pragma unroll
        for (int j = 0; j < 4; ++j)
            h[t][j] = __fadd_rn(__fmul_rn(__ldg(row + sx[j]), a0[j]), __fmul_rn(__ldg(row + sx1[j]), a1[j]));
    }
    const bool cols_inside = gq >= tx0 && gq + 3 < tx0 + out && gq + 3 < dst_w && gq >= 0;
#pragma unroll
    for (int k = 0; k < kPasteRows; ++k) {
        const int oy = 2 * a + k;
        const int gy = ty0 + oy;
        if (oy >= out || gy < 0 || gy >= dst_h) continue;
        // row taps: even rows (f = 0.75) blend source rows a+k/2-1, a+k/2; odd rows (f = 0.25) a+k/2, a+k/2+1;
        // the first and the last output row take one source row with weight 1 (the other tap has weight 0)
        const int t0 = (k >> 1) + (k & 1);                       // index into h[] of source row sy
        float b1 = (k & 1) ? 0.25f : 0.75f;
        if (oy == 0 || oy == out - 1) b1 = 0.f;
        const float b0 = 1.f - b1;
        float o[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const float h0 = (oy == 0) ? h[1][j] : h[t0][j];
            const float h1 = (oy == out - 1) ? h[t0][j] : h[t0 + 1][j];
            o[j] = __fadd_rn(__fmul_rn(h0, b0), __fmul_rn(h1, b1));
        }
        float* d = dst + (int64_t)gy * dst_w + gq;
        if (cols_inside && later == 0) {
            __stcs(reinterpret_cast<float4*>(d), make_float4(o[0], o[1], o[2], o[3]));
            continue;
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int gx = gq + j;
            bool owned = gx >= tx0 && gx < tx0 + out && gx >= 0 && gx < dst_w;
            for (unsigned mm = later; mm; mm &= mm - 1) {
                const int l = __ffs(mm) - 1;
                owned = owned && !(gy >= tiles.y[l] && gy < tiles.y[l] + out && gx >= tiles.x[l] && gx < tiles.x[l] + out);
            }
            if (owned) d[j] = o[j];
        }
    }
}

// ---- the blend of SURVEY.md 8d in ONE kernel ------------------------------------------------------------------------
// logits [V][Bt][S][S] -> de-augment + mean over the views + sigmoid + bilinear x2 + ownership test -> preds[H][W]:
// tta_merge64_kernel and paste_tiles_x2_kernel fused, bit-identical to running them one after the other, without the
// [B][S][S] probability intermediate.  One CTA = one 64 x 64 block of a tile's merged map = a 128 x 128 block of its
// window.  Two things make it cheaper than the pair: (1) a block whose whole window area a LATER tile covers returns
// before its first load -- with make_grid's overlaps that is half of all blocks, so half of the logits are never read;
// (2) the merged values go to the paste through shared memory.  The x2 filter needs one merged pixel of halo around
// the block: 260 pixels re-merged per CTA with scalar loads (+6 % of the reads, all L2 hits).
constexpr int kBlendP = kMergeTile + 2;          // merged block + halo
constexpr int kBlendPS = kMergeTile + 4;         // row stride of the shared tile (floats)

__global__ void __launch_bounds__(512, 2)
tta_blend_x2_kernel(const float* __restrict__ logits, int V, int Bt, int b0, int S, ViewMaps maps, PasteTiles tiles,
                    int first_tile, float* __restrict__ dst, int dst_h, int dst_w) {
    extern __shared__ __align__(16) float mtile[];      // [4][64][64] while merging, then the [66][68] merged tile
    constexpr int ROWS = 2;
    const int tid = threadIdx.x;
    const int l16 = tid & 15, rg = tid >> 4;
    const int b = b0 + blockIdx.z;                      // tile inside the logits batch
    const int tl = first_tile + blockIdx.z;             // tile inside the image's tile list
    const int I0 = blockIdx.y * kMergeTile, J0 = blockIdx.x * kMergeTile;
    const int out = 2 * S;
    const int ty0 = tiles.y[tl], tx0 = tiles.x[tl];
    // window area of this block in dst; later tiles that cover it completely / partly
    const int by0 = ty0 + 2 * I0, bx0 = tx0 + 2 * J0;
    unsigned later = 0;
    for (int l = tl + 1; l < tiles.n; ++l) {
        const int lx = tiles.x[l], ly = tiles.y[l];
        if (bx0 >= lx && bx0 + 2 * kMergeTile <= lx + out && by0 >= ly && by0 + 2 * kMergeTile <= ly + out) return;
        if (bx0 + 2 * kMergeTile > lx && bx0 < lx + out && by0 + 2 * kMergeTile > ly && by0 < ly + out) later |= 1u << l;
    }
    if (by0 >= dst_h || bx0 >= dst_w || by0 + 2 * kMergeTile <= 0 || bx0 + 2 * kMergeTile <= 0) return;

    // ---- merge of the 64 x 64 block: the body of tta_merge64_kernel<2, 2>
    constexpr int RSTEP = kMergeTile / ROWS;
    float4 acc[ROWS];
#pragma unroll
    for (int g = 0; g < 2; ++g) {
        if (g * 4 >= V) break;
        float4 val[4][ROWS];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int v = g * 4 + u;
            if (v >= V) continue;
            const int* m = maps.m[v];
            const float* src = logits + ((int64_t)v * Bt + b) * S * S;
            if (m[1] == 0) {
                const float* p = src + (m[4] > 0 ? J0 + 4 * l16 + m[5] : m[5] - J0 - 4 * l16 - 3);
#pragma unroll
                for (int r = 0; r < ROWS; ++r)
                    val[u][r] = __ldg(reinterpret_cast<const float4*>(p + (int64_t)(m[0] * (I0 + rg + RSTEP * r) + m[2]) * S));
            } else {
                const int row0 = m[1] > 0 ? J0 + m[2] : m[2] - J0 - (kMergeTile - 1);
                const int col0 = m[3] > 0 ? I0 + m[5] : m[5] - I0 - (kMergeTile - 1);
                const float* p = src + (int64_t)(row0 + rg) * S + col0 + 4 * l16;
#pragma unroll
                for (int r = 0; r < ROWS; ++r)
                    val[u][r] = __ldg(reinterpret_cast<const float4*>(p + (int64_t)(RSTEP * r) * S));
            }
        }
        if (g) __syncthreads();
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int v = g * 4 + u;
            if (v >= V || maps.m[v][1] == 0) continue;
            const int* m = maps.m[v];
            float* t = mtile + u * kMergeTile * kMergeTile;
#pragma unroll
            for (int r = 0; r < ROWS; ++r) {
                const int q = rg + RSTEP * r;
                const int jl = m[1] > 0 ? q : kMergeTile - 1 - q;
                const float e[4] = {val[u][r].x, val[u][r].y, val[u][r].z, val[u][r].w};
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const int il = m[3] > 0 ? 4 * l16 + k : kMergeTile - 1 - 4 * l16 - k;
                    t[il * kMergeTile + (jl ^ merge_swz(il))] = e[k];
                }
            }
        }
        __syncthreads();
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int v = g * 4 + u;
            if (v >= V) continue;
            const int* m = maps.m[v];
#pragma unroll
            for (int r = 0; r < ROWS; ++r) {
                float4 x = val[u][r];
                if (m[1] == 0) {
                    if (m[4] < 0) x = make_float4(x.w, x.z, x.y, x.x);
                } else {
                    const int il = rg + RSTEP * r;
                    const float4 w = *reinterpret_cast<const float4*>(mtile + u * kMergeTile * kMergeTile +
                                                                      il * kMergeTile + ((l16 ^ ((il >> 2) & 7)) << 2));
                    x = (il & 32) ? make_float4(w.z, w.w, w.x, w.y) : w;
                }
                if (v == 0) acc[r] = x;
                else { acc[r].x += x.x; acc[r].y += x.y; acc[r].z += x.z; acc[r].w += x.w; }
            }
        }
    }
    __syncthreads();                                    // every read of the transposition tiles is done: reuse the space
    float* P = mtile;                                   // P[(i - I0 + 1) * kBlendPS + (j - J0 + 1)]
    const float fv = (float)V;
#pragma unroll
    for (int r = 0; r < ROWS; ++r) {
        float4 o = make_float4(acc[r].x / fv, acc[r].y / fv, acc[r].z / fv, acc[r].w / fv);
        o = make_float4(sigmoidf_acc(o.x), sigmoidf_acc(o.y), sigmoidf_acc(o.z), sigmoidf_acc(o.w));
        float* pr = P + (rg + RSTEP * r + 1) * kBlendPS + 4 * l16 + 1;
        pr[0] = o.x; pr[1] = o.y; pr[2] = o.z; pr[3] = o.w;
    }
    // halo ring: rows I0-1 and I0+64 (66 pixels each), columns J0-1 and J0+64 (64 each); same sum order, same
    // division and sigmoid as above, so a halo pixel equals the value its own block computes
    if (tid < 2 * kBlendP + 2 * kMergeTile) {
        int li, lj;                                      // position in P
        if (tid < 2 * kBlendP) { li = tid < kBlendP ? 0 : kBlendP - 1; lj = tid % kBlendP; }
        else { const int t = tid - 2 * kBlendP; lj = t < kMergeTile ? 0 : kBlendP - 1; li = 1 + t % kMergeTile; }
        const int i = I0 + li - 1, j = J0 + lj - 1;
        if (i >= 0 && i < S && j >= 0 && j < S) {
            float sum = 0.f;
            for (int v = 0; v < V; ++v) {
                const int* m = maps.m[v];
                const float x = __ldg(logits + ((int64_t)v * Bt + b) * S * S + (int64_t)(m[0] * i + m[1] * j + m[2]) * S +
                                      (m[3] * i + m[4] * j + m[5]));
                sum = v == 0 ? x : sum + x;
            }
            P[li * kBlendPS + lj] = sigmoidf_acc(sum / fv);
        }
    }
    __syncthreads();

    // ---- x2 bilinear + ownership + store: paste_tiles_x2_kernel on the shared tile.  Items = (aligned quad of dst
    // columns, group of 8 output rows): 33 quads cover the 128 columns whatever the alignment of tx0.
    const int aq0 = bx0 & ~3;
    const int n_quads = (bx0 & 3) ? 33 : 32;
    for (int item = tid; item < n_quads * 16; item += 512) {
        const int q = item % n_quads, rgo = item / n_quads;
        const int gq = aq0 + 4 * q;
        if (gq >= dst_w || gq + 3 < 0) continue;
        const int a = I0 + rgo * 4;                      // output rows 2a .. 2a+7 of the tile
        const int gy_lo = ty0 + 2 * a;
        if (gy_lo >= dst_h || gy_lo + 7 < 0) continue;
        int lsx[4], lsx1[4];
        float a0[4], a1[4];
        bool col_ok[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int oxr = gq + j - tx0;                // column inside the tile's window
            col_ok[j] = oxr >= 2 * J0 && oxr < 2 * J0 + 2 * kMergeTile && gq + j >= 0 && gq + j < dst_w;
            const int ox = min(max(oxr, 2 * J0), 2 * J0 + 2 * kMergeTile - 1);
            int c = (ox >> 1) - ((ox & 1) ? 0 : 1);
            float f = (ox & 1) ? 0.25f : 0.75f;
            if (c < 0) { c = 0; f = 0.f; }
            if (c >= S - 1) { c = S - 1; f = 0.f; }
            lsx[j] = c - J0 + 1;
            lsx1[j] = min(c + 1, S - 1) - J0 + 1;
            a1[j] = f;
            a0[j] = 1.f - f;
        }
        float h[6][4];
#pragma unroll
        for (int t = 0; t < 6; ++t) {
            const float* row = P + (min(max(a - 1 + t, 0), S - 1) - I0 + 1) * kBlendPS;
#pragma unroll
            for (int j = 0; j < 4; ++j) h[t][j] = __fadd_rn(__fmul_rn(row[lsx[j]], a0[j]), __fmul_rn(row[lsx1[j]], a1[j]));
        }
        const bool quad_inside = col_ok[0] && col_ok[1] && col_ok[2] && col_ok[3];
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const int oy = 2 * a + k;
            const int gy = ty0 + oy;
            if (gy < 0 || gy >= dst_h) continue;
            const int t0 = (k >> 1) + (k & 1);
            float b1 = (k & 1) ? 0.25f : 0.75f;
            if (oy == 0 || oy == out - 1) b1 = 0.f;
            const float bb0 = 1.f - b1;
            float o[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const float h0 = (oy == 0) ? h[1][j] : h[t0][j];
                const float h1 = (oy == out - 1) ? h[t0][j] : h[t0 + 1][j];
                o[j] = __fadd_rn(__fmul_rn(h0, bb0), __fmul_rn(h1, b1));
            }
            float* d = dst + (int64_t)gy * dst_w + gq;
            if (quad_inside && later == 0) {
                __stcs(reinterpret_cast<float4*>(d), make_float4(o[0], o[1], o[2], o[3]));
                continue;
            }
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                bool owned = col_ok[j];
                const int gx = gq + j;
                for (unsigned mm = later; mm; mm &= mm - 1) {
                    const int l = __ffs(mm) - 1;
                    owned = owned && !(gy >= tiles.y[l] && gy < tiles.y[l] + out && gx >= tiles.x[l] && gx < tiles.x[l] + out);
                }
                if (owned) d[j] = o[j];
            }
        }
    }
}

// ---- opt-in: Gaussian overlap-tile blending (north_star "TTA views" bullet; NOT the reference's behaviour -- the
// reference overwrites, tta.py:213, and that stays the default and the parity mode) -------------------------------
// acc[gy][gx] += w * v, wsum[gy][gx] += w for ONE tile, v = the same bilinear x2 value the paste kernels write,
// w = g[oy] * g[ox] (separable window table of length 2S, built on the host).  Tiles are accumulated by successive
// launches in tile order, so the fp32 sums are deterministic; blend_finalize divides.
__global__ void __launch_bounds__(256)
blend_tile_gaussian_x2_kernel(const float* __restrict__ sp, int S, int ty0, int tx0, const float* __restrict__ g,
                              float* __restrict__ acc, float* __restrict__ wsum, int dst_h, int dst_w) {
    const int out = 2 * S;
    const int tid = threadIdx.y * blockDim.x + threadIdx.x;
    const int ox = blockIdx.x * kPasteBX + (tid & 63);
    const int gx = tx0 + ox;
    if (ox >= out || gx < 0 || gx >= dst_w) return;
    int sx = (ox >> 1) - ((ox & 1) ? 0 : 1);
    float a1 = (ox & 1) ? 0.25f : 0.75f;
    if (sx < 0) { sx = 0; a1 = 0.f; }
    if (sx >= S - 1) { sx = S - 1; a1 = 0.f; }
    const int sx1 = min(sx + 1, S - 1);
    const float a0 = 1.f - a1;
    const float wx = __ldg(g + ox);
    const int a = (blockIdx.y * kPasteBY + (tid >> 6) * 8) >> 1;
    float h[6];
#pragma unroll
    for (int t = 0; t < 6; ++t) {
        const float* row = sp + (int64_t)min(max(a - 1 + t, 0), S - 1) * S;
        h[t] = __fadd_rn(__fmul_rn(__ldg(row + sx), a0), __fmul_rn(__ldg(row + sx1), a1));
    }
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        const int oy = 2 * a + k;
        const int gy = ty0 + oy;
        if (oy >= out || gy < 0 || gy >= dst_h) continue;
        const int t0 = (k >> 1) + (k & 1);
        float b1 = (k & 1) ? 0.25f : 0.75f;
        if (oy == 0 || oy == out - 1) b1 = 0.f;
        const float h0 = (oy == 0) ? h[1] : h[t0];
        const float h1 = (oy == out - 1) ? h[t0] : h[t0 + 1];
        const float v = __fadd_rn(__fmul_rn(h0, 1.f - b1), __fmul_rn(h1, b1));
        const float w = __fmul_rn(__ldg(g + oy), wx);
        const int64_t idx = (int64_t)gy * dst_w + gx;
        acc[idx] = __fadd_rn(acc[idx], __fmul_rn(w, v));
        wsum[idx] = __fadd_rn(wsum[idx], w);
    }
}

__global__ void blend_finalize_kernel(const float* __restrict__ acc, const float* __restrict__ wsum, int64_t n,
                                      float* __restrict__ out) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const float w = wsum[i];
        out[i] = w > 0.f ? __fdiv_rn(acc[i], w) : 0.f;
    }
}

struct PreLut {
    float v[3][256];
};

// out[c][y][x] = lut[c][ (p00+p01+p10+p11+2) >> 2 ], window pixels outside the image read as 0.
__global__ void preprocess_tile_kernel(const uint8_t* __restrict__ img, int img_h, int img_w, int y0, int x0, int S,
                                       PreLut lut, float* __restrict__ out) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    const int y = blockIdx.y * blockDim.y + threadIdx.y;
    if (x >= S || y >= S) return;
    int sum[3] = {2, 2, 2};
#pragma unroll
    for (int dy = 0; dy < 2; ++dy)
#pragma unroll
        for (int dx = 0; dx < 2; ++dx) {
            const int iy = y0 + 2 * y + dy, ix = x0 + 2 * x + dx;
            if (iy >= 0 && iy < img_h && ix >= 0 && ix < img_w) {
                const uint8_t* p = img + ((int64_t)iy * img_w + ix) * 3;
                sum[0] += p[0];
                sum[1] += p[1];
                sum[2] += p[2];
            }
        }
    const int64_t plane = (int64_t)S * S;
    const int64_t o = (int64_t)y * S + x;
    out[o] = lut.v[0][sum[0] >> 2];
    out[plane + o] = lut.v[1][sum[1] >> 2];
    out[2 * plane + o] = lut.v[2][sum[2] >> 2];
}

}  // namespace eds

using namespace eds;

static int check_view_maps(const int* view_maps_host, int V, int S, ViewMaps* maps, const char* what) {
    for (int v = 0; v < V; ++v) {
        const int* m = view_maps_host + v * 6;
        // a signed permutation with offsets that keeps [0,S)^2 inside [0,S)^2
        const bool straight = m[1] == 0 && m[3] == 0 && (m[0] == 1 || m[0] == -1) && (m[4] == 1 || m[4] == -1);
        const bool swapped = m[0] == 0 && m[4] == 0 && (m[1] == 1 || m[1] == -1) && (m[3] == 1 || m[3] == -1);
        EDS_REQUIRE(straight || swapped, "%s: view %d map is not a flip/rot90", what, v);
        for (int corner = 0; corner < 4; ++corner) {
            const int i = (corner & 1) ? S - 1 : 0, j = (corner & 2) ? S - 1 : 0;
            const int r = m[0] * i + m[1] * j + m[2], c = m[3] * i + m[4] * j + m[5];
            EDS_REQUIRE(r >= 0 && r < S && c >= 0 && c < S, "%s: view %d map leaves the tile", what, v);
        }
        for (int q = 0; q < 6; ++q) maps->m[v][q] = m[q];
    }
    return EDS_OK;
}

// 16-byte vector loads of the 64 x 64 merge need S % 64 == 0 and column offsets that keep them aligned
static bool merge_vector_ok(const ViewMaps& maps, int V, int S, const void* a, const void* b) {
    bool vec = S % kMergeTile == 0 && (((uintptr_t)a | (uintptr_t)b) & 15) == 0;
    for (int v = 0; v < V && vec; ++v) {
        const int* m = maps.m[v];
        const int step = m[1] == 0 ? m[4] : m[3];
        vec = step > 0 ? m[5] % 4 == 0 : (m[5] + 1) % 4 == 0;
    }
    return vec;
}


extern "C" int eds_tta_merge(const float* logits, int V, int B, int S, const int* view_maps_host,
                             int apply_sigmoid, float* prob, void* stream) {
    EDS_REQUIRE(logits && prob && view_maps_host, "tta_merge: null pointer");
    EDS_REQUIRE(V >= 1 && V <= 8, "tta_merge: V=%d not in 1..8", V);
    EDS_REQUIRE(B >= 1 && B <= 65535 && S >= 1, "tta_merge: bad B=%d S=%d", B, S);
    ViewMaps maps;
    if (int rc = check_view_maps(view_maps_host, V, S, &maps, "tta_merge")) return rc;
    // 64x64 vector kernel when the tile size and every column offset keep the 16-byte loads aligned
    const bool vec = merge_vector_ok(maps, V, S, logits, prob);
    if (vec) {
        const int smem = 4 * kMergeTile * kMergeTile * (int)sizeof(float);
        // 512 threads x 2 rows measured best on B200 (50.0 us for 48 maps of 1024^2; 256 x 4 rows: 53.2 us;
        // 3 CTAs/SM at 80 registers spills: 59.4 us)
        auto kern = tta_merge64_kernel<2, 2>;
        static PerDevice once;
        if (int rc = smem_opt_in(once, kern, smem, "tta_merge")) return rc;
        dim3 grid(S / kMergeTile, S / kMergeTile, B);
        kern<<<grid, 512, smem, as_stream(stream)>>>(logits, V, B, S, maps, apply_sigmoid, prob);
        return check_launch("tta_merge64_kernel");
    }
    dim3 block(32, 8), grid(ceil_div(S, 32), ceil_div(S, 32), B);
    tta_merge_kernel<<<grid, block, 0, as_stream(stream)>>>(logits, V, B, S, maps, apply_sigmoid, prob);
    return check_launch("tta_merge_kernel");
}

extern "C" int eds_resize_paste_f32(const float* src, int src_h, int src_w, int crop_y, int crop_x, int crop_h,
                                    int crop_w, float* dst, int dst_h, int dst_w, int dst_y, int dst_x,
                                    int out_h, int out_w, void* stream) {
    EDS_REQUIRE(src && dst, "resize_paste: null pointer");
    EDS_REQUIRE(crop_h > 0 && crop_w > 0 && out_h > 0 && out_w > 0, "resize_paste: empty crop or output");
    EDS_REQUIRE(crop_y >= 0 && crop_x >= 0 && crop_y + crop_h <= src_h && crop_x + crop_w <= src_w,
                "resize_paste: crop [%d:%d,%d:%d] outside %dx%d source", crop_y, crop_y + crop_h, crop_x,
                crop_x + crop_w, src_h, src_w);
    dim3 block(64, 4), grid(ceil_div(out_w, kPasteBX), ceil_div(out_h, kPasteBY));
    resize_paste_kernel<<<grid, block, 0, as_stream(stream)>>>(src, src_w, crop_y, crop_x, crop_h, crop_w, dst,
                                                             dst_h, dst_w, dst_y, dst_x, out_h, out_w,
                                                             (double)crop_h / out_h, (double)crop_w / out_w);
    return check_launch("resize_paste_kernel");
}

static int paste_tiles_launch(const float* src, int n_src, int first_tile, int n_tiles, int S, const int* ys_host,
                              const int* xs_host, float* dst, int dst_h, int dst_w, void* stream) {
    EDS_REQUIRE(src && dst && ys_host && xs_host, "paste_tiles_x2: null pointer");
    EDS_REQUIRE(n_tiles >= 1 && n_tiles <= kPasteMaxTiles && S >= 1, "paste_tiles_x2: n_tiles=%d (1..%d), S=%d", n_tiles,
                kPasteMaxTiles, S);
    EDS_REQUIRE(n_src >= 1 && first_tile >= 0 && first_tile + n_src <= n_tiles,
                "paste_tiles_x2: tiles %d..%d outside the list of %d", first_tile, first_tile + n_src - 1, n_tiles);
    EDS_REQUIRE(dst_w % 4 == 0 && (((uintptr_t)dst) & 15) == 0, "paste_tiles_x2: dst rows must be 16-byte aligned "
                "(dst_w %% 4 == 0); use eds_resize_paste_f32 for other widths");
    PasteTiles tiles;
    tiles.n = n_tiles;
    for (int b = 0; b < kPasteMaxTiles; ++b) {
        tiles.y[b] = b < n_tiles ? ys_host[b] : 0;
        tiles.x[b] = b < n_tiles ? xs_host[b] : 0;
    }
    dim3 block(64, 4), grid(ceil_div(2 * S + 3, 4 * 64), ceil_div(2 * S, 4 * kPasteRows), n_src);
    paste_tiles_x2_kernel<<<grid, block, 0, as_stream(stream)>>>(src, S, tiles, first_tile, dst, dst_h, dst_w);
    return check_launch("paste_tiles_x2_kernel");
}

extern "C" int eds_paste_tiles_x2_f32(const float* src, int n_tiles, int S, const int* ys_host, const int* xs_host,
                                      float* dst, int dst_h, int dst_w, void* stream) {
    return paste_tiles_launch(src, n_tiles, 0, n_tiles, S, ys_host, xs_host, dst, dst_h, dst_w, stream);
}

extern "C" int eds_paste_tiles_owned_x2_f32(const float* src, int n_src, int first_tile, int n_tiles, int S,
                                            const int* ys_host, const int* xs_host, float* dst, int dst_h, int dst_w,
                                            void* stream) {
    return paste_tiles_launch(src, n_src, first_tile, n_tiles, S, ys_host, xs_host, dst, dst_h, dst_w, stream);
}

extern "C" int eds_tta_blend_supported(int V, int S, const int* view_maps_host, int dst_w) {
    if (V < 1 || V > 8 || S < kMergeTile || !view_maps_host || dst_w % 4 != 0) return 0;
    ViewMaps maps;
    if (check_view_maps(view_maps_host, V, S, &maps, "tta_blend") != EDS_OK) return 0;
    return merge_vector_ok(maps, V, S, nullptr, nullptr) ? 1 : 0;
}

extern "C" int eds_tta_blend_x2_f32(const float* logits, int V, int Bt, int b0, int n_src, int S,
                                    const int* view_maps_host, int first_tile, int n_tiles, const int* ys_host,
                                    const int* xs_host, float* dst, int dst_h, int dst_w, void* stream) {
    EDS_REQUIRE(logits && dst && view_maps_host && ys_host && xs_host, "tta_blend: null pointer");
    EDS_REQUIRE(V >= 1 && V <= 8, "tta_blend: V=%d not in 1..8", V);
    EDS_REQUIRE(Bt >= 1 && b0 >= 0 && n_src >= 1 && b0 + n_src <= Bt && n_src <= 65535, "tta_blend: tiles %d..%d outside "
                "the batch of %d", b0, b0 + n_src - 1, Bt);
    EDS_REQUIRE(n_tiles >= 1 && n_tiles <= kPasteMaxTiles && first_tile >= 0 && first_tile + n_src <= n_tiles,
                "tta_blend: tiles %d..%d outside the list of %d (max %d)", first_tile, first_tile + n_src - 1, n_tiles,
                kPasteMaxTiles);
    ViewMaps maps;
    if (int rc = check_view_maps(view_maps_host, V, S, &maps, "tta_blend")) return rc;
    EDS_REQUIRE(dst_w % 4 == 0 && merge_vector_ok(maps, V, S, logits, dst),
                "tta_blend: needs S %% 64 == 0, dst_w %% 4 == 0 and 16-byte aligned buffers (use eds_tta_merge + "
                "eds_paste_tiles_x2_f32 otherwise; eds_tta_blend_supported tells)");
    PasteTiles tiles;
    tiles.n = n_tiles;
    for (int b = 0; b < kPasteMaxTiles; ++b) {
        tiles.y[b] = b < n_tiles ? ys_host[b] : 0;
        tiles.x[b] = b < n_tiles ? xs_host[b] : 0;
    }
    const int smem = 4 * kMergeTile * kMergeTile * (int)sizeof(float);
    static PerDevice once;
    if (int rc = smem_opt_in(once, tta_blend_x2_kernel, smem, "tta_blend")) return rc;
    dim3 grid(S / kMergeTile, S / kMergeTile, n_src);
    tta_blend_x2_kernel<<<grid, 512, smem, as_stream(stream)>>>(logits, V, Bt, b0, S, maps, tiles, first_tile, dst, dst_h,
                                                              dst_w);
    return check_launch("tta_blend_x2_kernel");
}

extern "C" int eds_blend_tile_gaussian_x2_f32(const float* src, int S, int dst_y, int dst_x, const float* window,
                                              float* acc, float* wsum, int dst_h, int dst_w, void* stream) {
    EDS_REQUIRE(src && window && acc && wsum, "blend_tile_gaussian: null pointer");
    EDS_REQUIRE(S >= 1 && dst_h > 0 && dst_w > 0, "blend_tile_gaussian: bad sizes");
    dim3 block(64, 4), grid(ceil_div(2 * S, kPasteBX), ceil_div(2 * S, kPasteBY));
    blend_tile_gaussian_x2_kernel<<<grid, block, 0, as_stream(stream)>>>(src, S, dst_y, dst_x, window, acc, wsum, dst_h,
                                                                        dst_w);
    return check_launch("blend_tile_gaussian_x2_kernel");
}

extern "C" int eds_blend_finalize_f32(const float* acc, const float* wsum, int64_t n, float* out, void* stream) {
    EDS_REQUIRE(acc && wsum && out && n > 0, "blend_finalize: bad arguments");
    int64_t blocks = (n + 255) / 256;
    if (blocks > 148 * 16) blocks = 148 * 16;
    blend_finalize_kernel<<<(unsigned)blocks, 256, 0, as_stream(stream)>>>(acc, wsum, n, out);
    return check_launch("blend_finalize_kernel");
}

extern "C" int eds_preprocess_tile_u8(const uint8_t* img, int img_h, int img_w, int y0, int x0, int S,
                                      const double* mean3_host, const double* std3_host, float* out,
                                      void* stream) {
    EDS_REQUIRE(img && out && mean3_host && std3_host, "preprocess_tile: null pointer");
    EDS_REQUIRE(S > 0 && img_h > 0 && img_w > 0, "preprocess_tile: bad sizes");
    PreLut lut;
    for (int c = 0; c < 3; ++c)
        for (int v = 0; v < 256; ++v)
            // float64 arithmetic then one rounding, as numpy does for archs/__init__.py:88-97 + .float()
            lut.v[c][v] = (float)((((double)v / 255.0) - mean3_host[c]) / std3_host[c]);
    dim3 block(32, 8), grid(ceil_div(S, 32), ceil_div(S, 8));
    preprocess_tile_kernel<<<grid, block, 0, as_stream(stream)>>>(img, img_h, img_w, y0, x0, S, lut, out);
    return check_launch("preprocess_tile_kernel");
}
