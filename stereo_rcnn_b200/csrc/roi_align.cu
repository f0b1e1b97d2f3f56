// roi_align.cu -- RoIAlign forward / backward (reference layout) and the fused
// pyramid RoIAlign+average used by the product forward (sm_100a).
//
// Arithmetic follows lib/model/roi_align/src/roi_align_kernel.cu:27-68 exactly:
// fp32 roi scaling, fp64 for the sub-expressions the source writes with `1.` literals
// (roi size, bin size, tap weights), one fused multiply-add for the lattice coordinate,
// taps outside [0,H) x [0,W) -> 0, hstart = min(floor(h), H-2) (so [H-1,H) extrapolates).
//
// Kernels:
//  * roi_align_fwd_nchw  : drop-in for ROIAlignForward (NCHW in, R x C x ah x aw out).
//      Geometry is hoisted: one thread per (roi, tap, channel-run) instead of recomputing
//      9 divisions per output element; writes coalesced along (ph,pw).
//  * roi_align_bwd_nchw  : drop-in for ROIAlignBackward.
//  * roi_align_pyramid_nhwc: PyramidRoI_Feat (stereo_rcnn.py:110-139) in ONE launch for all
//      levels: level routing, per-level scale, (P+1)^2 tap lattice and the 2x2/stride-1
//      average of modules/roi_align.py:29, on NHWC features.  One CTA per (roi, output row):
//      two lattice rows are staged in shared memory (each tap = four coalesced 128-bit
//      channel-vector loads), then averaged and stored as coalesced channel vectors -- the
//      lattice (69 MB for the 14x14 keypoint pooling) never touches HBM.
#include <cuda_fp16.h>
#include <stdlib.h>

#include "common.cuh"

namespace {

struct RoiGeom {
    float start_w, start_h, bin_w, bin_h;
    int batch;
};

__device__ __forceinline__ RoiGeom roi_geom(const float* roi, float scale, int ah, int aw) {
    RoiGeom g;
    g.batch = (int)roi[0];
    float sw = __fmul_rn(roi[1], scale), sh = __fmul_rn(roi[2], scale);
    float ew = __fmul_rn(roi[3], scale), eh = __fmul_rn(roi[4], scale);
    float rw = fmaxf((float)((double)__fsub_rn(ew, sw) + 1.), 0.f);
    float rh = fmaxf((float)((double)__fsub_rn(eh, sh) + 1.), 0.f);
    g.bin_h = (float)((double)rh / ((double)ah - 1.));
    g.bin_w = (float)((double)rw / ((double)aw - 1.));
    g.start_w = sw;
    g.start_h = sh;
    return g;
}

struct Tap {
    int h0, w0;
    double w00, w01, w10, w11;
    bool zero;
};

__device__ __forceinline__ Tap make_tap(const RoiGeom& g, int ph, int pw, int H, int W) {
    Tap t;
    float h = __fmaf_rn((float)ph, g.bin_h, g.start_h);
    float w = __fmaf_rn((float)pw, g.bin_w, g.start_w);
    t.h0 = (int)fminf(floorf(h), (float)(H - 2));
    t.w0 = (int)fminf(floorf(w), (float)(W - 2));
    t.zero = (h < 0 || h >= H || w < 0 || w >= W);
    double hr = (double)__fsub_rn(h, (float)t.h0), wr = (double)__fsub_rn(w, (float)t.w0);
    t.w00 = (1. - hr) * (1. - wr);
    t.w01 = (1. - hr) * wr;
    t.w10 = hr * (1. - wr);
    t.w11 = hr * wr;
    return t;
}

// double evaluation order of the source: ((a*(1-hr))*(1-wr) + (b*(1-hr))*wr) + ...
__device__ __forceinline__ float tap_value(const Tap& t, float a, float b, float c, float d, double hr_unused = 0) {
    (void)hr_unused;
    double v = (double)a * t.w00 + (double)b * t.w01 + (double)c * t.w10 + (double)d * t.w11;
    return (float)v;
}

__global__ void __launch_bounds__(256)
roi_align_fwd_nchw(const float* __restrict__ feat, int C, int H, int W, const float* __restrict__ rois,
                   int ah, int aw, float scale, float* __restrict__ out) {
    // grid: (roi, channel-chunk); threads sweep (c, ph, pw) with pw fastest
    const int n = blockIdx.x;
    const RoiGeom g = roi_geom(rois + 5 * n, scale, ah, aw);
    const int taps = ah * aw;
    const int c0 = blockIdx.y * 32;
    const int cend = min(c0 + 32, C);
    for (int e = threadIdx.x; e < (cend - c0) * taps; e += blockDim.x) {
        int c = c0 + e / taps, p = e % taps;
        int ph = p / aw, pw = p % aw;
        Tap t = make_tap(g, ph, pw, H, W);
        float v = 0.f;
        if (!t.zero) {
            const float* f = feat + (((size_t)g.batch * C + c) * H + t.h0) * W + t.w0;
            v = tap_value(t, f[0], f[1], f[W], f[W + 1]);
        }
        out[((size_t)n * C + c) * taps + p] = v;
    }
}

__global__ void __launch_bounds__(256)
roi_align_bwd_nchw(const float* __restrict__ top, int C, int H, int W, const float* __restrict__ rois,
                   int ah, int aw, float scale, float* __restrict__ bottom) {
    const int n = blockIdx.x;
    const RoiGeom g = roi_geom(rois + 5 * n, scale, ah, aw);
    const int taps = ah * aw;
    const int c0 = blockIdx.y * 32;
    const int cend = min(c0 + 32, C);
    for (int e = threadIdx.x; e < (cend - c0) * taps; e += blockDim.x) {
        int c = c0 + e / taps, p = e % taps;
        int ph = p / aw, pw = p % aw;
        Tap t = make_tap(g, ph, pw, H, W);
        if (t.zero) continue;
        double tv = (double)top[((size_t)n * C + c) * taps + p];
        float* b = bottom + (((size_t)g.batch * C + c) * H + t.h0) * W + t.w0;
        atomicAdd(b, (float)(tv * t.w00));
        atomicAdd(b + 1, (float)(tv * t.w01));
        atomicAdd(b + W, (float)(tv * t.w10));
        atomicAdd(b + W + 1, (float)(tv * t.w11));
    }
}

// ---- deterministic backward (SURVEY 7.8): the same scatter, accumulated in 64-bit FIXED POINT.  Integer addition is
// associative, so the result does not depend on the order in which the atomics land (nor on the order of the RoIs):
// bit-identical run to run, which the reference's float atomicAdds (roi_align_kernel.cu:132-139) are not.
// Scale 2^e with e chosen from max|top_grad| so that 2^20 contributions of that magnitude cannot overflow 2^62: the
// quantum is max|top| * 2^-41, far below fp32 resolution of the sum.
__global__ void __launch_bounds__(256)
absmax_kernel(const float* __restrict__ x, size_t n, unsigned* __restrict__ out) {
    unsigned m = 0u;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const unsigned b = __float_as_uint(x[i]) & 0x7fffffffu;        // |x| as bits: monotonic for finite / inf
        m = b > m ? b : m;
    }
    m = __reduce_max_sync(0xffffffffu, m);
    if ((threadIdx.x & 31) == 0 && m) atomicMax(out, m);
}

__device__ __forceinline__ int fixed_exponent(unsigned absmax_bits) {
    if (absmax_bits == 0u || absmax_bits >= 0x7f800000u) return 0;    // all zero, or inf / nan: nothing sensible to scale
    int ex;
    frexpf(__uint_as_float(absmax_bits), &ex);                         // |x| < 2^ex
    return 41 - ex;                                                    // |x| * 2^e < 2^41; 2^20 of them < 2^61
}

__global__ void __launch_bounds__(256)
roi_align_bwd_fixed_kernel(const float* __restrict__ top, int C, int H, int W, const float* __restrict__ rois, int ah,
                           int aw, float scale, const unsigned* __restrict__ absmax,
                           unsigned long long* __restrict__ acc) {
    const int n = blockIdx.x;
    const RoiGeom g = roi_geom(rois + 5 * n, scale, ah, aw);
    const double s = ldexp(1.0, fixed_exponent(*absmax));
    const int taps = ah * aw;
    const int c0 = blockIdx.y * 32;
    const int cend = min(c0 + 32, C);
    for (int e = threadIdx.x; e < (cend - c0) * taps; e += blockDim.x) {
        int c = c0 + e / taps, p = e % taps;
        int ph = p / aw, pw = p % aw;
        Tap t = make_tap(g, ph, pw, H, W);
        if (t.zero) continue;
        const double tv = (double)top[((size_t)n * C + c) * taps + p] * s;
        unsigned long long* b = acc + (((size_t)g.batch * C + c) * H + t.h0) * W + t.w0;
        atomicAdd(b, (unsigned long long)__double2ll_rn(tv * t.w00));         // two's complement: wraps like int64
        atomicAdd(b + 1, (unsigned long long)__double2ll_rn(tv * t.w01));
        atomicAdd(b + W, (unsigned long long)__double2ll_rn(tv * t.w10));
        atomicAdd(b + W + 1, (unsigned long long)__double2ll_rn(tv * t.w11));
    }
}

__global__ void __launch_bounds__(256)
fixed_to_float_kernel(const unsigned long long* __restrict__ acc, size_t n, const unsigned* __restrict__ absmax,
                      float* __restrict__ out) {
    const double inv = ldexp(1.0, -fixed_exponent(*absmax));
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
        out[i] = (float)((double)(long long)acc[i] * inv);
}

struct PyramidArgs {
    const float* feat[4];
    int H[4], W[4];
    float scale[4];
};

// stereo_rcnn.py:113-119: round(ln(sqrt(h*w)/224) + 4) clamped to [2,5] (fp32, natural log)
__device__ __forceinline__ int roi_level(const float* roi) {
    float h = __fadd_rn(__fsub_rn(roi[4], roi[2]), 1.0f);
    float w = __fadd_rn(__fsub_rn(roi[3], roi[1]), 1.0f);
    float l = logf(__fdiv_rn(sqrtf(__fmul_rn(h, w)), 224.0f));
    l = rintf(__fadd_rn(l, 4.0f));  // torch.round: half to even
    l = fminf(fmaxf(l, 2.f), 5.f);
    return (int)l - 2;
}

// the geometry of one lattice tap of a pyramid RoI on NHWC features (forward and backward share it)
struct TapRec {
    double w00, w01, w10, w11;
    long long off;      // element offset of the top-left source pixel, or -1 for a zero tap
};

__device__ __forceinline__ TapRec tap_record(const RoiGeom& g, int ph, int pw, int H, int W, int C) {
    const Tap t = make_tap(g, ph, pw, H, W);
    TapRec tr;
    tr.w00 = t.w00; tr.w01 = t.w01; tr.w10 = t.w10; tr.w11 = t.w11;
    tr.off = t.zero ? -1 : (long long)((((size_t)g.batch * H + t.h0) * W + t.w0) * C);
    return tr;
}

// One CTA per (roi, block of RB output rows); C % 4 == 0.  The CTA walks the RB+1 lattice rows of its block with a
// rolling pair of rows in shared memory (each lattice row is built once per CTA instead of once per output row: at
// RB = 7 the 14x14 pooling does 8/7 instead of 2x the tap work), and the tap geometry -- fp64 weights, offsets -- is
// built once per (row, column) by the first threads instead of once per channel vector.
// dynamic smem = 2 * (P+1) * C floats for the lattice rows + (RB+1) * (P+1) tap records.

__global__ void __launch_bounds__(256)
roi_align_pyramid_nhwc(PyramidArgs a, int C, const float* __restrict__ rois, int P, int RB,
                       float* __restrict__ out, int out_ld, int out_coff, int round_tf32) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int L = P + 1;
    const int C4 = C >> 2;
    float4* lat = reinterpret_cast<float4*>(smem_raw);                               // [2][L][C4]
    TapRec* taps = reinterpret_cast<TapRec*>(smem_raw + (size_t)2 * L * C4 * sizeof(float4));   // [RB+1][L]
    const int n = blockIdx.x, ph0 = blockIdx.y * RB;
    const int rows = min(RB, P - ph0);                 // output rows of this CTA
    const float* roi = rois + 5 * n;
    const int lv = roi_level(roi);
    const int H = a.H[lv], W = a.W[lv];
    const float* __restrict__ feat = a.feat[lv];
    const RoiGeom g = roi_geom(roi, a.scale[lv], L, L);
    for (int e = threadIdx.x; e < (rows + 1) * L; e += blockDim.x) {
        const int r = e / L, pw = e - r * L;
        taps[e] = tap_record(g, ph0 + r, pw, H, W, C);
    }
    __syncthreads();
    const size_t wstep = (size_t)W * C4;
    for (int r = 0; r <= rows; ++r) {
        float4* cur = lat + (size_t)(r & 1) * L * C4;
        for (int e = threadIdx.x; e < L * C4; e += blockDim.x) {
            const int c4 = e % C4, pw = e / C4;
            const TapRec& t = taps[r * L + pw];
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (t.off >= 0) {
                const float4* f00 = reinterpret_cast<const float4*>(feat + t.off) + c4;
                const float4 p00 = __ldg(f00), p01 = __ldg(f00 + C4);
                const float4 p10 = __ldg(f00 + wstep), p11 = __ldg(f00 + wstep + C4);
                v.x = (float)((double)p00.x * t.w00 + (double)p01.x * t.w01 + (double)p10.x * t.w10 + (double)p11.x * t.w11);
                v.y = (float)((double)p00.y * t.w00 + (double)p01.y * t.w01 + (double)p10.y * t.w10 + (double)p11.y * t.w11);
                v.z = (float)((double)p00.z * t.w00 + (double)p01.z * t.w01 + (double)p10.z * t.w10 + (double)p11.z * t.w11);
                v.w = (float)((double)p00.w * t.w00 + (double)p01.w * t.w01 + (double)p10.w * t.w10 + (double)p11.w * t.w11);
            }
            cur[e] = v;
        }
        __syncthreads();
        if (r == 0) continue;
        const float4* top = lat + (size_t)((r - 1) & 1) * L * C4;
        const int ph = ph0 + r - 1;
        float* orow = out + ((size_t)n * P + ph) * P * out_ld + out_coff;
        for (int e = threadIdx.x; e < P * C4; e += blockDim.x) {
            const int c4 = e % C4, pw = e / C4;
            const float4 a0 = top[pw * C4 + c4], a1 = top[(pw + 1) * C4 + c4];
            const float4 b0 = cur[pw * C4 + c4], b1 = cur[(pw + 1) * C4 + c4];
            float4 o;  // avg_pool2d(2, stride 1): ((a+b)+(c+d)) * 0.25
            o.x = __fmul_rn(__fadd_rn(__fadd_rn(a0.x, a1.x), __fadd_rn(b0.x, b1.x)), 0.25f);
            o.y = __fmul_rn(__fadd_rn(__fadd_rn(a0.y, a1.y), __fadd_rn(b0.y, b1.y)), 0.25f);
            o.z = __fmul_rn(__fadd_rn(__fadd_rn(a0.z, a1.z), __fadd_rn(b0.z, b1.z)), 0.25f);
            o.w = __fmul_rn(__fadd_rn(__fadd_rn(a0.w, a1.w), __fadd_rn(b0.w, b1.w)), 0.25f);
            if (round_tf32 == 2) {      // fp16 output for the kind::f16 convs (same element strides, half the bytes)
                __half2 lo = __floats2half2_rn(o.x, o.y), hi = __floats2half2_rn(o.z, o.w);
                uint2 pk;
                pk.x = *reinterpret_cast<uint32_t*>(&lo);
                pk.y = *reinterpret_cast<uint32_t*>(&hi);
                __half* ob = reinterpret_cast<__half*>(out) + ((size_t)n * P + ph) * P * out_ld + out_coff;
                *reinterpret_cast<uint2*>(ob + (size_t)pw * out_ld + 4 * c4) = pk;
                continue;
            }
            if (round_tf32) {   // the pooled tile is read only by tensor-core convs: make TF32 truncation exact
                o.x = sb_round_tf32(o.x); o.y = sb_round_tf32(o.y); o.z = sb_round_tf32(o.z); o.w = sb_round_tf32(o.w);
            }
            *reinterpret_cast<float4*>(orow + (size_t)pw * out_ld + 4 * c4) = o;
        }
        __syncthreads();       // the next lattice row overwrites `top`
    }
}

// ---- adjoint of roi_align_pyramid_nhwc, deterministic: the fixed-point scatter of roi_align_bwd_fixed_kernel on the
// forward's routing and tap geometry.  Lattice point (i, j) feeds the output cells (i-1..i, j-1..j) of the 2x2 average
// with weight 1/4 each, so its gradient is 1/4 of the sum of those cells' gradients (fp64, fixed order); it then goes
// to the tap's four source pixels with the tap's fp64 weights.  One CTA per RoI; threads sweep (tap, channel) with the
// channel fastest, so the 64-bit atomics of a warp hit consecutive words.
struct PyramidGradArgs {
    unsigned long long* acc[4];
    int H[4], W[4];
    float scale[4];
};

__global__ void __launch_bounds__(256)
absmax_rows_kernel(const float* __restrict__ x, size_t rows, int cols, int ld, unsigned* __restrict__ out) {
    unsigned m = 0u;
    const size_t n = rows * (size_t)cols;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const size_t r = i / (size_t)cols, c = i - r * (size_t)cols;
        const unsigned b = __float_as_uint(x[r * (size_t)ld + c]) & 0x7fffffffu;
        m = b > m ? b : m;
    }
    m = __reduce_max_sync(0xffffffffu, m);
    if ((threadIdx.x & 31) == 0 && m) atomicMax(out, m);
}

__global__ void __launch_bounds__(256)
roi_align_pyramid_nhwc_bwd_fixed(PyramidGradArgs a, int N, int C, const float* __restrict__ rois, int P,
                                 const float* __restrict__ top, int top_ld, const unsigned* __restrict__ absmax) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    TapRec* taps = reinterpret_cast<TapRec*>(smem_raw);      // [L][L]
    const int L = P + 1;
    const int n = blockIdx.x;
    const float* roi = rois + 5 * n;
    const int lv = roi_level(roi);
    const int H = a.H[lv], W = a.W[lv];
    const RoiGeom g = roi_geom(roi, a.scale[lv], L, L);
    if (g.batch < 0 || g.batch >= N) return;      // no image of the batch: nothing to scatter (whole CTA leaves)
    for (int e = threadIdx.x; e < L * L; e += blockDim.x) taps[e] = tap_record(g, e / L, e % L, H, W, C);
    __syncthreads();
    const double s = ldexp(1.0, fixed_exponent(*absmax));
    const float* __restrict__ tg = top + (size_t)n * P * P * top_ld;
    unsigned long long* __restrict__ acc = a.acc[lv];
    const size_t wstep = (size_t)W * C;
    for (int e = threadIdx.x; e < L * L * C; e += blockDim.x) {
        const int t = e / C, c = e - t * C;
        const TapRec& tr = taps[t];
        if (tr.off < 0) continue;
        const int i = t / L, j = t - i * L;
        double gs = 0.;
        for (int oh = i - 1; oh <= i; ++oh) {
            if (oh < 0 || oh >= P) continue;
            if (j >= 1) gs += (double)tg[((size_t)oh * P + j - 1) * top_ld + c];
            if (j < P) gs += (double)tg[((size_t)oh * P + j) * top_ld + c];
        }
        if (gs == 0.) continue;
        const double tv = 0.25 * gs * s;
        unsigned long long* b = acc + tr.off + c;
        atomicAdd(b, (unsigned long long)__double2ll_rn(tv * tr.w00));       // two's complement: wraps like int64
        atomicAdd(b + C, (unsigned long long)__double2ll_rn(tv * tr.w01));
        atomicAdd(b + wstep, (unsigned long long)__double2ll_rn(tv * tr.w10));
        atomicAdd(b + wstep + C, (unsigned long long)__double2ll_rn(tv * tr.w11));
    }
}

// stereo_rcnn.py:128: scale = feat.size(2) / im_info[0][0] (python float), then float(...)
float pyramid_scale(int height, float im_h) { return (float)((double)height / (double)im_h); }

}  // namespace

extern "C" int sb_roi_align_forward(const float* features, int N, int C, int H, int W, const float* rois,
                                    int R, int ah, int aw, float spatial_scale, float* out,
                                    sb_stream_t stream) {
    (void)N;
    if (R == 0) return SB_OK;
    if (R < 0 || C <= 0 || ah < 2 || aw < 2 || !features || !rois || !out) return SB_EINVAL;
    dim3 grid(R, (C + 31) / 32);
    roi_align_fwd_nchw<<<grid, 256, 0, sb_cs(stream)>>>(features, C, H, W, rois, ah, aw, spatial_scale, out);
    SB_LAUNCHED();
    SB_CHECK_LAUNCH();
    return SB_OK;
}

extern "C" int sb_roi_align_backward(const float* top_grad, int N, int C, int H, int W, const float* rois,
                                     int R, int ah, int aw, float spatial_scale, float* bottom_grad,
                                     sb_stream_t stream) {
    (void)N;
    if (R == 0) return SB_OK;
    if (R < 0 || C <= 0 || ah < 2 || aw < 2 || !top_grad || !rois || !bottom_grad) return SB_EINVAL;
    dim3 grid(R, (C + 31) / 32);
    roi_align_bwd_nchw<<<grid, 256, 0, sb_cs(stream)>>>(top_grad, C, H, W, rois, ah, aw, spatial_scale, bottom_grad);
    SB_LAUNCHED();
    SB_CHECK_LAUNCH();
    return SB_OK;
}

extern "C" size_t sb_roi_align_backward_det_workspace(int N, int C, int H, int W) {
    if (N < 1 || C < 1 || H < 2 || W < 2) return 0;
    return (size_t)N * C * H * W * 8 + 16;
}

extern "C" int sb_roi_align_backward_det(const float* top_grad, int N, int C, int H, int W, const float* rois, int R,
                                         int ah, int aw, float spatial_scale, float* bottom_grad, void* workspace,
                                         size_t workspace_bytes, sb_stream_t stream) {
    if (R < 0 || N < 1 || C <= 0 || H < 2 || W < 2 || ah < 2 || aw < 2 || !top_grad || !rois || !bottom_grad || !workspace ||
        workspace_bytes < sb_roi_align_backward_det_workspace(N, C, H, W) || (reinterpret_cast<uintptr_t>(workspace) & 7))
        return SB_EINVAL;
    cudaStream_t st = sb_cs(stream);
    const size_t n = (size_t)N * C * H * W;
    unsigned long long* acc = static_cast<unsigned long long*>(workspace);
    unsigned* absmax = reinterpret_cast<unsigned*>(acc + n);
    cudaError_t e = cudaMemsetAsync(workspace, 0, n * 8 + 16, st);
    if (e != cudaSuccess) return (int)e;
    const size_t nt = (size_t)R * C * ah * aw;
    if (R > 0) {
        absmax_kernel<<<(int)((nt + 255) / 256 < 1184 ? (nt + 255) / 256 : 1184), 256, 0, st>>>(top_grad, nt, absmax);
        SB_LAUNCHED();
        dim3 grid(R, (C + 31) / 32);
        roi_align_bwd_fixed_kernel<<<grid, 256, 0, st>>>(top_grad, C, H, W, rois, ah, aw, spatial_scale, absmax, acc);
        SB_LAUNCHED();
    }
    fixed_to_float_kernel<<<(int)((n + 255) / 256 < 2368 ? (n + 255) / 256 : 2368), 256, 0, st>>>(acc, n, absmax, bottom_grad);
    SB_LAUNCHED();
    SB_CHECK_LAUNCH();
    return SB_OK;
}

extern "C" int sb_roi_align_pyramid_nhwc(const float* const* feats, const int* heights, const int* widths,
                                         int C, float im_h, const float* rois, int R, int pooled,
                                         float* out, int out_ld, int out_coff, int round_tf32,
                                         sb_stream_t stream) {
    if (R == 0) return SB_OK;
    if (R < 0 || (C & 3) || pooled < 1 || (out_ld & 3) || (out_coff & 3)) return SB_EINVAL;
    PyramidArgs a;
    for (int l = 0; l < 4; ++l) {
        a.feat[l] = feats[l];
        a.H[l] = heights[l];
        a.W[l] = widths[l];
        a.scale[l] = pyramid_scale(heights[l], im_h);
    }
    // output rows per CTA: all of a 7x7 tile (8 lattice rows for 7 outputs), half of a 14x14 tile
    int RB = pooled <= 8 ? pooled : (pooled + 1) / 2;
    static const int rb_env = getenv("SB_ROI_RB") ? atoi(getenv("SB_ROI_RB")) : 0;     // A/B knob (tools/ab.sh)
    if (rb_env > 0) RB = rb_env < pooled ? rb_env : pooled;
    size_t smem = (size_t)2 * (pooled + 1) * C * sizeof(float) + (size_t)(RB + 1) * (pooled + 1) * sizeof(TapRec);
    if (smem > 200 * 1024) return SB_EINVAL;
    static size_t cur_max_dev[kSbMaxDevices] = {0};
    size_t& cur_max = cur_max_dev[sb_cur_device()];
    if (cur_max == 0) cur_max = 48 * 1024;
    if (smem > cur_max) {
        cudaFuncSetAttribute(roi_align_pyramid_nhwc, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        cur_max = smem;
    }
    dim3 grid(R, (pooled + RB - 1) / RB);
    roi_align_pyramid_nhwc<<<grid, 256, smem, sb_cs(stream)>>>(a, C, rois, pooled, RB, out, out_ld, out_coff, round_tf32);
    SB_LAUNCHED();
    SB_CHECK_LAUNCH();
    return SB_OK;
}

extern "C" size_t sb_roi_align_pyramid_nhwc_backward_workspace(int N, const int* heights, const int* widths, int C) {
    if (N < 1 || C < 1 || !heights || !widths) return 0;
    size_t n = 0;
    for (int l = 0; l < 4; ++l) {
        if (heights[l] < 2 || widths[l] < 2) return 0;
        n += (size_t)N * heights[l] * widths[l] * C;
    }
    return n * 8 + 16;
}

extern "C" int sb_roi_align_pyramid_nhwc_backward(const float* top_grad, int top_ld, int top_coff, int C, float im_h,
                                                  const float* rois, int R, int pooled, int N, const int* heights,
                                                  const int* widths, float* const* grad_feats, void* workspace,
                                                  size_t workspace_bytes, sb_stream_t stream) {
    if (R < 0 || C < 4 || (C & 3) || pooled < 1 || N < 1 || top_coff < 0 || top_ld < top_coff + C || !heights ||
        !widths || !grad_feats || (R > 0 && (!top_grad || !rois)) || !workspace || (reinterpret_cast<uintptr_t>(workspace) & 7))
        return SB_EINVAL;
    const size_t need = sb_roi_align_pyramid_nhwc_backward_workspace(N, heights, widths, C);
    if (need == 0 || workspace_bytes < need) return SB_EINVAL;
    for (int l = 0; l < 4; ++l)
        if (!grad_feats[l]) return SB_EINVAL;
    const int L = pooled + 1;
    const size_t smem = (size_t)L * L * sizeof(TapRec);
    if (smem > 48 * 1024) return SB_EINVAL;
    PyramidGradArgs a;
    size_t cnt[4], off = 0;
    unsigned long long* acc = static_cast<unsigned long long*>(workspace);
    for (int l = 0; l < 4; ++l) {
        cnt[l] = (size_t)N * heights[l] * widths[l] * C;
        a.acc[l] = acc + off;
        off += cnt[l];
        a.H[l] = heights[l];
        a.W[l] = widths[l];
        a.scale[l] = pyramid_scale(heights[l], im_h);
    }
    unsigned* absmax = reinterpret_cast<unsigned*>(acc + off);
    cudaStream_t st = sb_cs(stream);
    cudaError_t e = cudaMemsetAsync(workspace, 0, need, st);
    if (e != cudaSuccess) return (int)e;
    if (R > 0) {
        const size_t rows = (size_t)R * pooled * pooled, nt = rows * C;
        absmax_rows_kernel<<<(int)((nt + 255) / 256 < 1184 ? (nt + 255) / 256 : 1184), 256, 0, st>>>(
            top_grad + top_coff, rows, C, top_ld, absmax);
        SB_LAUNCHED();
        roi_align_pyramid_nhwc_bwd_fixed<<<R, 256, smem, st>>>(a, N, C, rois, pooled, top_grad + top_coff, top_ld, absmax);
        SB_LAUNCHED();
    }
    for (int l = 0; l < 4; ++l) {
        const size_t n = cnt[l];
        fixed_to_float_kernel<<<(int)((n + 255) / 256 < 2368 ? (n + 255) / 256 : 2368), 256, 0, st>>>(a.acc[l], n, absmax,
                                                                                                     grad_feats[l]);
        SB_LAUNCHED();
    }
    SB_CHECK_LAUNCH();
    return SB_OK;
}
