// Axial attention core for the MHSA encoder blocks and the MHCA skip gates.
//
// Reference: src/main/archs/axial_attention_v2.py:178-213 (AxialAttention.forward) and
// :100-135 (CrossAxialAttention.forward) after the to_qvk / to_kq / to_v projections
// (those are 1x1 convolutions and run on the conv kernels with their BatchNorm1d folded).
// Everything from the relative-position einsums to out_norm is one kernel:
//   sim[d][j] = s_qr * sum_i q[i][d] rq[i][d-j+L-1] + s_kr * sum_i k[i][d] rk[i][d-j+L-1]
//             + s_dots * sum_i q[i][d] k[i][j]              (attention_norm: scale only, its
//                                                             per-channel shift cancels in softmax)
//   attn = softmax_j(sim)
//   y[h*dv+i][d] = a_kv * sum_j attn[d][j] rv[i][d-j+L-1] + c_kv + a_out * sum_j attn[d][j] v[i][j] + c_out
// One CTA handles one (sequence, head); sequences are rows or columns of the NHWC map,
// addressed by stride so no rearrange / permute is ever materialised.
#include "common.cuh"

namespace eds {

constexpr int kAttnThreads = 256;

template <typename T>
__global__ void __launch_bounds__(kAttnThreads)
axial_attention_kernel(const T* __restrict__ qk, int qk_cstride, const T* __restrict__ vsrc, int v_cstride, int H,
                       int W, int axis, int heads, int dqk, int dv, const float* __restrict__ rel,
                       const float* __restrict__ sim_scale, const float* __restrict__ out_scale,
                       const float* __restrict__ out_shift, int relu, T* __restrict__ y) {
    extern __shared__ float sm[];
    const int L = axis == 0 ? H : W;
    const int R = 2 * L - 1;
    float* s_q = sm;                    // [dqk][L]
    float* s_k = s_q + dqk * L;         // [dqk][L]
    float* s_vT = s_k + dqk * L;        // [L][dv]
    float* s_rq = s_vT + L * dv;        // [dqk][R]
    float* s_rk = s_rq + dqk * R;       // [dqk][R]
    float* s_rv = s_rk + dqk * R;       // [dv][R]
    float* s_att = s_rv + dv * R;       // [L][L+1]

    const int tid = threadIdx.x;
    const int head = blockIdx.y;
    const int seq = blockIdx.x;
    // pixel index of position d of this sequence
    int64_t pix0, pstride;
    if (axis == 0) {
        const int n = seq / W, wq = seq % W;
        pix0 = (int64_t)n * H * W + wq;
        pstride = W;
    } else {
        pix0 = (int64_t)seq * W;  // seq = n*H + h
        pstride = 1;
    }
    const int G = 2 * dqk + (vsrc ? 0 : dv);

    for (int idx = tid; idx < L * G; idx += kAttnThreads) {
        const int d = idx / G, c = idx % G;
        const float val = Elem<T>::ld(qk + (pix0 + (int64_t)d * pstride) * qk_cstride + head * G + c);
        if (c < dqk) s_q[c * L + d] = val;
        else if (c < 2 * dqk) s_k[(c - dqk) * L + d] = val;
        else s_vT[d * dv + (c - 2 * dqk)] = val;
    }
    if (vsrc)
        for (int idx = tid; idx < L * dv; idx += kAttnThreads) {
            const int d = idx / dv, c = idx % dv;
            s_vT[d * dv + c] = Elem<T>::ld(vsrc + (pix0 + (int64_t)d * pstride) * v_cstride + head * dv + c);
        }
    for (int idx = tid; idx < dqk * R; idx += kAttnThreads) {
        s_rq[idx] = rel[idx];
        s_rk[idx] = rel[dqk * R + idx];
    }
    for (int idx = tid; idx < dv * R; idx += kAttnThreads) s_rv[idx] = rel[2 * dqk * R + idx];
    __syncthreads();

    const float a_qr = sim_scale[head * 3 + 0], a_kr = sim_scale[head * 3 + 1], a_dots = sim_scale[head * 3 + 2];
    for (int idx = tid; idx < L * L; idx += kAttnThreads) {
        const int d = idx / L, j = idx % L;
        const int rpos = d - j + L - 1;
        float qr = 0.f, kr = 0.f, dots = 0.f;
        for (int i = 0; i < dqk; ++i) {
            const float qd = s_q[i * L + d];
            qr += qd * s_rq[i * R + rpos];
            kr += s_k[i * L + d] * s_rk[i * R + rpos];
            dots += qd * s_k[i * L + j];
        }
        s_att[d * (L + 1) + j] = a_qr * qr + a_kr * kr + a_dots * dots;
    }
    __syncthreads();

    const int lane = tid & 31, warp = tid >> 5;
    for (int d = warp; d < L; d += kAttnThreads / 32) {
        float* row = s_att + d * (L + 1);
        float mx = -3.4e38f;
        for (int j = lane; j < L; j += 32) mx = fmaxf(mx, row[j]);
        mx = warp_max(mx);
        float sum = 0.f;
        for (int j = lane; j < L; j += 32) {
            const float e = expf(row[j] - mx);
            row[j] = e;
            sum += e;
        }
        sum = warp_sum(sum);
        const float inv = 1.f / sum;
        for (int j = lane; j < L; j += 32) row[j] *= inv;
    }
    __syncthreads();

    const int CO = heads * dv;
    for (int idx = tid; idx < L * dv; idx += kAttnThreads) {
        const int d = idx / dv, i = idx % dv;
        const float* row = s_att + d * (L + 1);
        const float* rv = s_rv + i * R + d + L - 1;
        float out = 0.f, kv = 0.f;
        for (int j = 0; j < L; ++j) {
            const float a = row[j];
            out += a * s_vT[j * dv + i];
            kv += a * rv[-j];
        }
        const int ch = head * dv + i;
        const float r = (out_scale[ch] * kv + out_shift[ch]) + (out_scale[CO + ch] * out + out_shift[CO + ch]);
        Elem<T>::st(y + (pix0 + (int64_t)d * pstride) * CO + ch, relu ? fmaxf(r, 0.f) : r);
    }
}

int axial_attention_mma_try(const void* qk, int qk_cstride, const void* v, int v_cstride, int N, int H, int W, int axis,
                            int heads, int dqk, int dv, const float* rel, const float* sim_scale,
                            const float* out_scale, const float* out_shift, int relu, void* y, cudaStream_t stream);

}  // namespace eds

using namespace eds;

extern "C" int eds_axial_attention(const void* qk, int qk_cstride, const void* v, int v_cstride, int N, int H, int W,
                                   int axis, int heads, int dqk, int dv, const float* rel, const float* sim_scale,
                                   const float* out_scale, const float* out_shift, int relu, void* y,
                                   int dtype, void* stream) {
    EDS_REQUIRE(qk && rel && sim_scale && out_scale && out_shift && y, "axial_attention: null pointer");
    EDS_REQUIRE(axis == 0 || axis == 1, "axial_attention: axis=%d", axis);
    EDS_REQUIRE(N > 0 && H > 0 && W > 0 && heads > 0 && dqk > 0 && dv > 0, "axial_attention: bad shape");
    // bf16 activations: tensor-core kernel (attention_mma.cu); fp32 parity mode and shapes outside it
    // (dqk != 8, heads % 4 != 0, L > 64) run the CUDA-core kernel below.
    if (dtype == EDS_BF16) {
        const int rc = axial_attention_mma_try(qk, qk_cstride, v, v_cstride, N, H, W, axis, heads, dqk, dv, rel,
                                               sim_scale, out_scale, out_shift, relu, y, as_stream(stream));
        if (rc <= 0) return rc;
    }
    const int L = axis == 0 ? H : W;
    const int R = 2 * L - 1;
    const size_t smem = sizeof(float) * ((size_t)2 * dqk * L + (size_t)L * dv + (size_t)2 * dqk * R + (size_t)dv * R +
                                         (size_t)L * (L + 1));
    EDS_REQUIRE(smem <= 227 * 1024, "axial_attention: L=%d dv=%d needs %zu B shared memory (> 227 KB)", L, dv, smem);
    const int n_seq = axis == 0 ? N * W : N * H;
    EDS_REQUIRE(heads <= 65535, "axial_attention: heads=%d", heads);
    dim3 grid(n_seq, heads);
    cudaError_t e = cudaSuccess;
    EDS_DISPATCH_DTYPE(dtype, T, {
        if (smem > 48 * 1024)
            e = cudaFuncSetAttribute(axial_attention_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     (int)smem);
        if (e == cudaSuccess)
            axial_attention_kernel<T><<<grid, kAttnThreads, smem, as_stream(stream)>>>(
                (const T*)qk, qk_cstride, (const T*)v, v_cstride, H, W, axis, heads, dqk, dv, rel, sim_scale,
                out_scale, out_shift, relu, (T*)y);
    });
    if (e != cudaSuccess) {
        set_error("axial_attention: shared-memory opt-in failed: %s", cudaGetErrorString(e));
        return EDS_ERR_CUDA;
    }
    return check_launch("axial_attention_kernel");
}
