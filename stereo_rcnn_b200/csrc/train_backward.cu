// train_backward.cu -- the small kernels of the box-head training step (resnet.py:256-263,282-285,345-348 RCNN_top and
// the three linears; stereo_rcnn.py:248-257): dropout after the two ReLUs of RCNN_top, the backward of the tail
// linears, the "mask, scale and convert" step that turns an fp32 gradient into a tensor-core operand, and the permute
// of the fc6 weight gradient into the reference's [Cout][C][7][7] layout.  The two big products of each layer go
// through sb_gemm_tc.  Every reduction has a fixed order: the gradients are bit-identical run to run.
#include <cuda_fp16.h>

#include "common.cuh"

namespace {

// nn.Dropout(p = 0.2) with explicit random words: keep if word >= 0.2 * 2^32 (= 858993459.2), scale 1 / 0.8
constexpr unsigned kKeepFrom = 858993460u;

__device__ __forceinline__ bool kept(unsigned w) { return w >= kKeepFrom; }

__global__ void __launch_bounds__(256)
dropout_kernel(const float* __restrict__ x, const unsigned* __restrict__ words, size_t n, float* __restrict__ out32,
               __half* __restrict__ out16) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const float v = kept(words[i]) ? x[i] * 1.25f : 0.f;
        if (out32) out32[i] = v;
        if (out16) out16[i] = __float2half_rn(v);
    }
}

// d x[r][k] = sum_o d_out[r][o] W[o][k] over the 12 nc outputs of the tail (o < nc: cls, < 7nc: bbox, else dim)
__global__ void __launch_bounds__(256)
tail_dx_kernel(const float* __restrict__ d_cls, const float* __restrict__ d_box, const float* __restrict__ d_dim,
               int R, int K, int nc, const float* __restrict__ w_cls, const float* __restrict__ w_box,
               const float* __restrict__ w_dim, float* __restrict__ dx) {
    const size_t n = (size_t)R * K;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const int r = (int)(i / K), k = (int)(i - (size_t)r * K);
        float s = 0.f;
        for (int o = 0; o < nc; ++o) s = fmaf(d_cls[(size_t)r * nc + o], __ldg(w_cls + (size_t)o * K + k), s);
        for (int o = 0; o < 6 * nc; ++o) s = fmaf(d_box[(size_t)r * 6 * nc + o], __ldg(w_box + (size_t)o * K + k), s);
        for (int o = 0; o < 5 * nc; ++o) s = fmaf(d_dim[(size_t)r * 5 * nc + o], __ldg(w_dim + (size_t)o * K + k), s);
        dx[i] = s;
    }
}

// dW[o][k] = sum_r d_out[r][o] x[r][k] (k < K) and db[o] = sum_r d_out[r][o] (k == K), r in order
__global__ void __launch_bounds__(256)
tail_dw_kernel(const float* __restrict__ d_cls, const float* __restrict__ d_box, const float* __restrict__ d_dim,
               const float* __restrict__ x, int R, int K, int nc, float* __restrict__ dw_cls, float* __restrict__ db_cls,
               float* __restrict__ dw_box, float* __restrict__ db_box, float* __restrict__ dw_dim,
               float* __restrict__ db_dim) {
    const int o = blockIdx.y;
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k > K) return;
    const float* d;
    int ld, oo;
    float *dw, *db;
    if (o < nc) { d = d_cls; ld = nc; oo = o; dw = dw_cls; db = db_cls; }
    else if (o < 7 * nc) { d = d_box; ld = 6 * nc; oo = o - nc; dw = dw_box; db = db_box; }
    else { d = d_dim; ld = 5 * nc; oo = o - 7 * nc; dw = dw_dim; db = db_dim; }
    float s = 0.f;
    if (k < K) {
        for (int r = 0; r < R; ++r) s = fmaf(__ldg(d + (size_t)r * ld + oo), x[(size_t)r * K + k], s);
        dw[(size_t)oo * K + k] = s;
    } else {
        for (int r = 0; r < R; ++r) s += __ldg(d + (size_t)r * ld + oo);
        db[oo] = s;
    }
}

// ---- mask, scale and convert: g = dy * keep * 1.25 * (y > 0) (dropout after ReLU; y = the ReLU output), the bias
// gradient db = sum_r g (fixed order: 32-row partial sums, then the partials in order), and an fp16 copy of g times
// 2^e, e chosen on the device from max|g| so that the largest element lands in [2^14, 2^15): RCNN gradients are
// divided by the number of sampled RoIs and would otherwise flush in fp16.  inv_scale = 2^-e feeds sb_gemm_tc's alpha.
constexpr int kRowChunk = 32;

__global__ void __launch_bounds__(256)
mask_grad_kernel(const float* __restrict__ dy, const float* __restrict__ y, const unsigned* __restrict__ words, int R,
                 int C, float* __restrict__ g, float* __restrict__ part, unsigned* __restrict__ absmax) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    const int r0 = blockIdx.y * kRowChunk;
    unsigned m = 0u;
    if (c < C) {
        float s = 0.f;
        const int r1 = min(r0 + kRowChunk, R);
        for (int r = r0; r < r1; ++r) {
            const size_t i = (size_t)r * C + c;
            const float v = (kept(words[i]) && y[i] > 0.f) ? dy[i] * 1.25f : 0.f;
            g[i] = v;
            s += v;
            const unsigned b = __float_as_uint(v) & 0x7fffffffu;
            m = b > m ? b : m;
        }
        part[(size_t)blockIdx.y * C + c] = s;
    }
    m = __reduce_max_sync(0xffffffffu, m);
    if ((threadIdx.x & 31) == 0 && m) atomicMax(absmax, m);         // max is order independent
}

__device__ __forceinline__ int grad_exponent(unsigned absmax_bits) {
    if (absmax_bits == 0u || absmax_bits >= 0x7f800000u) return 0;
    int ex;
    frexpf(__uint_as_float(absmax_bits), &ex);                       // max|g| < 2^ex
    return max(-120, min(120, 15 - ex));                             // max|g| * 2^e in [2^14, 2^15)
}

__global__ void __launch_bounds__(256)
bias_sum_kernel(const float* __restrict__ part, int chunks, int C, const unsigned* __restrict__ absmax,
                float* __restrict__ db, float* __restrict__ inv_scale) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c < C && db) {
        float s = 0.f;
        for (int q = 0; q < chunks; ++q) s += part[(size_t)q * C + c];
        db[c] = s;
    }
    if (c == 0) *inv_scale = ldexpf(1.f, -grad_exponent(*absmax));
}

__global__ void __launch_bounds__(256)
scale_half_kernel(const float* __restrict__ g, size_t n, const unsigned* __restrict__ absmax, __half* __restrict__ g16) {
    const float s = ldexpf(1.f, grad_exponent(*absmax));
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
        g16[i] = __float2half_rn(g[i] * s);                          // exact scaling by a power of two, one rounding
}

// packed [Co][P][C] ((ph, pw, c) order of the NHWC pooled tile) -> [Co][C][P] (Conv2d weight [Co][C][7][7])
__global__ void __launch_bounds__(256)
permute_pc_kernel(const float* __restrict__ in, int Co, int P, int C, float* __restrict__ out) {
    const size_t n = (size_t)Co * P * C;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const size_t co = i / ((size_t)P * C);
        const int rem = (int)(i - co * P * C), c = rem / P, p = rem - c * P;
        out[i] = in[(co * P + p) * C + c];
    }
}

// the same through shared memory, one CTA per (co, 32 channels): reads of 32 consecutive channels per tap, writes of
// 32 x P consecutive floats (C % 32 == 0)
__global__ void __launch_bounds__(256)
permute_pc_tiled_kernel(const float* __restrict__ in, int P, int C, float* __restrict__ out) {
    extern __shared__ float tile[];                                  // [P][33]
    const size_t co = blockIdx.x;
    const int c0 = blockIdx.y * 32;
    for (int e = threadIdx.x; e < P * 32; e += blockDim.x) {
        const int p = e >> 5, cc = e & 31;
        tile[p * 33 + cc] = in[(co * P + p) * C + c0 + cc];
    }
    __syncthreads();
    float* o = out + (co * C + c0) * P;
    for (int e = threadIdx.x; e < P * 32; e += blockDim.x) {
        const int cc = e / P, p = e - cc * P;
        o[e] = tile[p * 33 + cc];
    }
}

int grid_for(size_t n) { return (int)((n + 255) / 256 < 4736 ? (n + 255) / 256 : 4736); }

}  // namespace

extern "C" int sb_dropout(const float* x, const unsigned* words, int R, int C, float* out32, void* out16,
                          sb_stream_t stream) {
    if (R < 0 || C < 1 || (R > 0 && (!x || !words || (!out32 && !out16)))) return SB_EINVAL;
    if (R == 0) return SB_OK;
    const size_t n = (size_t)R * C;
    dropout_kernel<<<grid_for(n), 256, 0, sb_cs(stream)>>>(x, words, n, out32, static_cast<__half*>(out16));
    SB_LAUNCHED();
    SB_CHECK_LAUNCH();
    return SB_OK;
}

extern "C" int sb_box_tail_backward(const float* d_cls, const float* d_bbox, const float* d_dim, const float* fc7, int R,
                                    int K, int n_classes, const float* w_cls, const float* w_box, const float* w_dim,
                                    float* d_fc7, float* dw_cls, float* db_cls, float* dw_box, float* db_box,
                                    float* dw_dim, float* db_dim, sb_stream_t stream) {
    if (R < 1 || K < 1 || n_classes < 1 || n_classes > 4 || !d_cls || !d_bbox || !d_dim || !fc7 || !w_cls || !w_box ||
        !w_dim || !d_fc7 || !dw_cls || !db_cls || !dw_box || !db_box || !dw_dim || !db_dim)
        return SB_EINVAL;
    cudaStream_t st = sb_cs(stream);
    tail_dx_kernel<<<grid_for((size_t)R * K), 256, 0, st>>>(d_cls, d_bbox, d_dim, R, K, n_classes, w_cls, w_box, w_dim,
                                                            d_fc7);
    SB_LAUNCHED();
    tail_dw_kernel<<<dim3(sb_div_up(K + 1, 256), 12 * n_classes), 256, 0, st>>>(d_cls, d_bbox, d_dim, fc7, R, K,
                                                                                 n_classes, dw_cls, db_cls, dw_box,
                                                                                 db_box, dw_dim, db_dim);
    SB_LAUNCHED();
    SB_CHECK_LAUNCH();
    return SB_OK;
}

extern "C" size_t sb_dropout_backward_workspace(int R, int C) {
    if (R < 1 || C < 1) return 0;
    return (size_t)R * C * 4 + (size_t)sb_div_up(R, kRowChunk) * C * 4 + 16;
}

extern "C" int sb_dropout_backward(const float* dy, const float* y, const unsigned* words, int R, int C, float* db,
                                   void* g16, float* inv_scale, void* workspace, size_t workspace_bytes,
                                   sb_stream_t stream) {
    if (R < 1 || C < 1 || !dy || !y || !words || !g16 || !inv_scale || !workspace ||
        workspace_bytes < sb_dropout_backward_workspace(R, C) || (reinterpret_cast<uintptr_t>(workspace) & 15))
        return SB_EINVAL;
    cudaStream_t st = sb_cs(stream);
    const int chunks = sb_div_up(R, kRowChunk);
    float* g = static_cast<float*>(workspace);
    float* part = g + (size_t)R * C;
    unsigned* absmax = reinterpret_cast<unsigned*>(part + (size_t)chunks * C);
    cudaError_t e = cudaMemsetAsync(absmax, 0, 4, st);
    if (e != cudaSuccess) return (int)e;
    mask_grad_kernel<<<dim3(sb_div_up(C, 256), chunks), 256, 0, st>>>(dy, y, words, R, C, g, part, absmax);
    SB_LAUNCHED();
    bias_sum_kernel<<<sb_div_up(C, 256), 256, 0, st>>>(part, chunks, C, absmax, db, inv_scale);
    SB_LAUNCHED();
    const size_t n = (size_t)R * C;
    scale_half_kernel<<<grid_for(n), 256, 0, st>>>(g, n, absmax, static_cast<__half*>(g16));
    SB_LAUNCHED();
    SB_CHECK_LAUNCH();
    return SB_OK;
}

extern "C" int sb_permute_pc_to_cp(const float* in, int Co, int P, int C, float* out, sb_stream_t stream) {
    if (Co < 1 || P < 1 || C < 1 || !in || !out) return SB_EINVAL;
    const size_t n = (size_t)Co * P * C;
    const size_t smem = (size_t)P * 33 * sizeof(float);
    if (C % 32 == 0 && smem <= 48 * 1024)
        permute_pc_tiled_kernel<<<dim3(Co, C / 32), 256, smem, sb_cs(stream)>>>(in, P, C, out);
    else
        permute_pc_kernel<<<grid_for(n), 256, 0, sb_cs(stream)>>>(in, Co, P, C, out);
    SB_LAUNCHED();
    SB_CHECK_LAUNCH();
    return SB_OK;
}
