// misc.cu -- small memory-bound layer ops of the Stereo R-CNN forward (sm_100a):
// max-pool, stride-2 subsample, keypoint-head tail, box-head tail, test-time decode.
#include <cuda_fp16.h>

#include "common.cuh"

unsigned long long g_sb_launches = 0;

extern "C" unsigned long long sb_launch_count(void) { return g_sb_launches; }
extern "C" int sb_version(void) { return 100; }
extern "C" int sb_device_cc(void) {
    cudaDeviceProp p;
    if (cudaGetDeviceProperties(&p, sb_cur_device()) != cudaSuccess) return -1;
    return p.major * 10 + p.minor;
}

namespace {

__global__ void __launch_bounds__(256)
fill_kernel(float4* __restrict__ p, size_t n4, float v) {
    size_t i = (size_t)blockIdx.x * 256 + threadIdx.x;
    const size_t stride = (size_t)gridDim.x * 256;
    const float4 f = make_float4(v, v, v, v);
    for (; i < n4; i += stride) p[i] = f;
}

// nn.MaxPool2d(kernel_size=3, stride=2, padding=0, ceil_mode=True) (resnet.py:113), NHWC
__global__ void __launch_bounds__(256)
maxpool_kernel(const float4* __restrict__ in, int N, int H, int W, int C4, int Ho, int Wo,
               float4* __restrict__ out) {
    const long long total = (long long)N * Ho * Wo * C4;
    long long e = (long long)blockIdx.x * 256 + threadIdx.x;
    if (e >= total) return;
    const int c = (int)(e % C4);
    long long t = e / C4;
    const int wo = (int)(t % Wo); t /= Wo;
    const int ho = (int)(t % Ho);
    const int n = (int)(t / Ho);
    float4 m = make_float4(-INFINITY, -INFINITY, -INFINITY, -INFINITY);
    for (int r = 0; r < 3; ++r) {
        const int hi = ho * 2 + r;
        if (hi >= H) break;
        for (int s = 0; s < 3; ++s) {
            const int wi = wo * 2 + s;
            if (wi >= W) break;
            const float4 v = __ldg(in + (((long long)n * H + hi) * W + wi) * C4 + c);
            m.x = fmaxf(m.x, v.x); m.y = fmaxf(m.y, v.y); m.z = fmaxf(m.z, v.z); m.w = fmaxf(m.w, v.w);
        }
    }
    out[e] = m;
}

// fp16 twin of maxpool_kernel: 8 channels (one 16-byte vector) per thread
__global__ void __launch_bounds__(256)
maxpool16_kernel(const uint4* __restrict__ in, int N, int H, int W, int C8, int Ho, int Wo, uint4* __restrict__ out) {
    const long long total = (long long)N * Ho * Wo * C8;
    long long e = (long long)blockIdx.x * 256 + threadIdx.x;
    if (e >= total) return;
    const int c = (int)(e % C8);
    long long t = e / C8;
    const int wo = (int)(t % Wo); t /= Wo;
    const int ho = (int)(t % Ho);
    const int n = (int)(t / Ho);
    const __half2 ninf = __float2half2_rn(-INFINITY);
    __half2 m0 = ninf, m1 = ninf, m2 = ninf, m3 = ninf;
    for (int r = 0; r < 3; ++r) {
        const int hi = ho * 2 + r;
        if (hi >= H) break;
        for (int s = 0; s < 3; ++s) {
            const int wi = wo * 2 + s;
            if (wi >= W) break;
            const uint4 v = __ldg(in + (((long long)n * H + hi) * W + wi) * C8 + c);
            m0 = __hmax2(m0, *reinterpret_cast<const __half2*>(&v.x));
            m1 = __hmax2(m1, *reinterpret_cast<const __half2*>(&v.y));
            m2 = __hmax2(m2, *reinterpret_cast<const __half2*>(&v.z));
            m3 = __hmax2(m3, *reinterpret_cast<const __half2*>(&v.w));
        }
    }
    uint4 o;
    o.x = *reinterpret_cast<uint32_t*>(&m0); o.y = *reinterpret_cast<uint32_t*>(&m1);
    o.z = *reinterpret_cast<uint32_t*>(&m2); o.w = *reinterpret_cast<uint32_t*>(&m3);
    out[e] = o;
}

__global__ void __launch_bounds__(256)
subsample2_kernel(const float4* __restrict__ in, int N, int H, int W, int C4, int Ho, int Wo,
                  float4* __restrict__ out) {
    const long long total = (long long)N * Ho * Wo * C4;
    long long e = (long long)blockIdx.x * 256 + threadIdx.x;
    if (e >= total) return;
    const int c = (int)(e % C4);
    long long t = e / C4;
    const int wo = (int)(t % Wo); t /= Wo;
    const int ho = (int)(t % Ho);
    const int n = (int)(t / Ho);
    out[e] = __ldg(in + (((long long)n * H + 2 * ho) * W + 2 * wo) * C4 + c);
}

// keypoint tail (stereo_rcnn.py:262-271): x [R,G,G,C] -> sum over height -> 1x1 conv C->6 -> [R,6,G]
// (kernel 1: grid (R, 4 column groups), one thread per channel: 4x the CTAs of a per-RoI mapping so that
// the 241 MB read runs with enough loads in flight), then softmax(4G), softmax(G), softmax(G) (kernel 2).
__device__ __forceinline__ float ld_as_float(const float* p) { return __ldg(p); }
__device__ __forceinline__ float ld_as_float(const __half* p) { return __half2float(__ldg(p)); }

template <typename T>
__global__ void __launch_bounds__(256)
kpts_colsum_kernel(const T* __restrict__ x, int G, int C, int cols_per_cta, const float* __restrict__ w,
                   const float* __restrict__ b, float* __restrict__ pred_all) {
    __shared__ float part[8 * 6];
    const int r = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int nw = blockDim.x >> 5;
    const T* xr = x + (size_t)r * G * G * C;
    const int col0 = blockIdx.y * cols_per_cta, col1 = min(G, col0 + cols_per_cta);
    for (int col = col0; col < col1; ++col) {
        float p[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
        for (int c = tid; c < C; c += blockDim.x) {
            float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
            int h = 0;
            for (; h + 3 < G; h += 4) {
                s0 += ld_as_float(xr + ((size_t)(h + 0) * G + col) * C + c);
                s1 += ld_as_float(xr + ((size_t)(h + 1) * G + col) * C + c);
                s2 += ld_as_float(xr + ((size_t)(h + 2) * G + col) * C + c);
                s3 += ld_as_float(xr + ((size_t)(h + 3) * G + col) * C + c);
            }
            for (; h < G; ++h) s0 += ld_as_float(xr + ((size_t)h * G + col) * C + c);
            const float s = (s0 + s1) + (s2 + s3);
#pragma unroll
            for (int j = 0; j < 6; ++j) p[j] = fmaf(w[j * C + c], s, p[j]);
        }
#pragma unroll
        for (int j = 0; j < 6; ++j) {
            float s = warp_sum(p[j]);
            if (lane == 0) part[warp * 6 + j] = s;
        }
        __syncthreads();
        if (tid < 6) {
            float s = 0.f;
            for (int q = 0; q < nw; ++q) s += part[q * 6 + tid];
            pred_all[((size_t)r * 6 + tid) * G + col] = s + (float)G * b[tid];
        }
        __syncthreads();
    }
}

// fp16 input: one warp per column, one 16-byte vector (8 channels) per lane and row; C == 256
__global__ void __launch_bounds__(256)
kpts_colsum16_kernel(const __half* __restrict__ x, int G, int C, const float* __restrict__ w,
                     const float* __restrict__ b, float* __restrict__ pred_all) {
    const int r = blockIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int col = blockIdx.y * 8 + warp;
    if (col >= G) return;
    const uint4* xr = reinterpret_cast<const uint4*>(x + (size_t)r * G * G * C) + lane;
    const int C8 = C >> 3;
    float s[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll 4
    for (int h = 0; h < G; ++h) {
        const uint4 v = __ldg(xr + ((size_t)h * G + col) * C8);
        const float2 f0 = __half22float2(*reinterpret_cast<const __half2*>(&v.x));
        const float2 f1 = __half22float2(*reinterpret_cast<const __half2*>(&v.y));
        const float2 f2 = __half22float2(*reinterpret_cast<const __half2*>(&v.z));
        const float2 f3 = __half22float2(*reinterpret_cast<const __half2*>(&v.w));
        s[0] += f0.x; s[1] += f0.y; s[2] += f1.x; s[3] += f1.y;
        s[4] += f2.x; s[5] += f2.y; s[6] += f3.x; s[7] += f3.y;
    }
#pragma unroll
    for (int j = 0; j < 6; ++j) {
        const float* wj = w + j * C + lane * 8;
        float p = 0.f;
#pragma unroll
        for (int e = 0; e < 8; ++e) p = fmaf(wj[e], s[e], p);
        p = warp_sum(p);
        if (lane == 0) pred_all[((size_t)r * 6 + j) * G + col] = p + (float)G * b[j];
    }
}

__global__ void __launch_bounds__(96)
kpts_softmax_kernel(const float* __restrict__ pred_all, int G, float* __restrict__ kpts_prob,
                    float* __restrict__ left_prob, float* __restrict__ right_prob) {
    const int r = blockIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const float* ka = pred_all + (size_t)r * 6 * G;
    const int n = warp == 0 ? 4 * G : G;
    const float* src = warp == 0 ? ka : ka + (3 + warp) * G;
    float* dst = warp == 0 ? kpts_prob + (size_t)r * 4 * G : (warp == 1 ? left_prob : right_prob) + (size_t)r * G;
    float m = -INFINITY;
    for (int e = lane; e < n; e += 32) m = fmaxf(m, src[e]);
    m = warp_max(m);
    float s = 0.f;
    for (int e = lane; e < n; e += 32) s += expf(src[e] - m);
    s = warp_sum(s);
    for (int e = lane; e < n; e += 32) dst[e] = expf(src[e] - m) / s;
}

// box tail (stereo_rcnn.py:253-257): three linears on fc7 + softmax over classes
// LOGITS = false: softmax probabilities (test time, sb_box_tail); true: the raw class scores (sb_box_tail_logits, the
// training forward: the cross entropy of sb_rcnn_loss takes logits)
template <bool LOGITS>
__global__ void __launch_bounds__(256)
box_tail_kernel(const float* __restrict__ fc7, int K, int nc, const float* __restrict__ w_cls,
                const float* __restrict__ b_cls, const float* __restrict__ w_box,
                const float* __restrict__ b_box, const float* __restrict__ w_dim,
                const float* __restrict__ b_dim, float* __restrict__ cls_prob,
                float* __restrict__ bbox_pred, float* __restrict__ dim_orien) {
    __shared__ float part[8][48];
    __shared__ float outv[48];
    const int r = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int n_out = 12 * nc;   // nc + 6nc + 5nc
    const float* f = fc7 + (size_t)r * K;
    for (int o = 0; o < n_out; ++o) {
        const float* w = o < nc ? w_cls + (size_t)o * K
                       : (o < 7 * nc ? w_box + (size_t)(o - nc) * K : w_dim + (size_t)(o - 7 * nc) * K);
        float s = 0.f;
        for (int k = tid; k < K; k += 256) s = fmaf(f[k], __ldg(w + k), s);
        s = warp_sum(s);
        if (lane == 0) part[warp][o] = s;
    }
    __syncthreads();
    if (tid < n_out) {
        float s = 0.f;
        for (int q = 0; q < 8; ++q) s += part[q][tid];
        s += tid < nc ? b_cls[tid] : (tid < 7 * nc ? b_box[tid - nc] : b_dim[tid - 7 * nc]);
        outv[tid] = s;
    }
    __syncthreads();
    if (LOGITS && tid < nc) cls_prob[(size_t)r * nc + tid] = outv[tid];
    if (!LOGITS && tid == 0) {
        float m = -INFINITY, s = 0.f;
        for (int j = 0; j < nc; ++j) m = fmaxf(m, outv[j]);
        for (int j = 0; j < nc; ++j) s += expf(outv[j] - m);
        for (int j = 0; j < nc; ++j) cls_prob[(size_t)r * nc + j] = expf(outv[j] - m) / s;
    }
    if (tid >= nc && tid < 7 * nc) bbox_pred[(size_t)r * 6 * nc + tid - nc] = outv[tid];
    if (tid >= 7 * nc && tid < n_out) dim_orien[(size_t)r * 5 * nc + tid - 7 * nc] = outv[tid];
}

// test_net.py:138-212 for one image; one thread per RoI
__global__ void __launch_bounds__(128)
test_decode_kernel(const float* __restrict__ rois_l, const float* __restrict__ rois_r,
                   const float* __restrict__ bbox_pred, const float* __restrict__ dim_orien,
                   const float* __restrict__ kpts_prob, const float* __restrict__ left_prob,
                   const float* __restrict__ right_prob, const float* __restrict__ im_info, int R, int nc,
                   int grid, float* __restrict__ pbl, float* __restrict__ pbr, float* __restrict__ dimo,
                   float* __restrict__ pkpts, const float* __restrict__ cls_prob, float* __restrict__ record,
                   int rec_ld) {
    const int r = blockIdx.x * 128 + threadIdx.x;
    if (r >= R) return;
    const float stds[4] = {0.1f, 0.1f, 0.2f, 0.2f};           // cfg.TRAIN.BBOX_NORMALIZE_STDS/MEANS
    const float dmean[5] = {1.6f, 1.5f, 4.0f, 0.0f, 0.0f};    // cfg.TRAIN.DIM_NORMALIZE_MEANS (STDS = 0.5)
    const float imh = im_info[0], imw = im_info[1], sc = im_info[2];
    const float xmax = __fsub_rn(imw, 1.0f), ymax = __fsub_rn(imh, 1.0f);
    const float4 bl = make_float4(rois_l[5 * r + 1], rois_l[5 * r + 2], rois_l[5 * r + 3], rois_l[5 * r + 4]);
    const float4 br = make_float4(rois_r[5 * r + 1], rois_r[5 * r + 2], rois_r[5 * r + 3], rois_r[5 * r + 4]);
    for (int j = 0; j < nc; ++j) {
        const float* d = bbox_pred + (size_t)r * 6 * nc + 6 * j;
        float dl[4] = {d[0], d[1], d[2], d[3]}, dr[4] = {d[4], d[1], d[5], d[3]};
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            dl[q] = __fadd_rn(__fmul_rn(dl[q], stds[q]), 0.0f);
            dr[q] = __fadd_rn(__fmul_rn(dr[q], stds[q]), 0.0f);
        }
        float4 a = sb_decode_clip(bl, dl[0], dl[1], dl[2], dl[3], xmax, ymax);
        float4 b = sb_decode_clip(br, dr[0], dr[1], dr[2], dr[3], xmax, ymax);
        float* o = pbl + (size_t)r * 4 * nc + 4 * j;
        o[0] = __fdiv_rn(a.x, sc); o[1] = __fdiv_rn(a.y, sc); o[2] = __fdiv_rn(a.z, sc); o[3] = __fdiv_rn(a.w, sc);
        o = pbr + (size_t)r * 4 * nc + 4 * j;
        o[0] = __fdiv_rn(b.x, sc); o[1] = __fdiv_rn(b.y, sc); o[2] = __fdiv_rn(b.z, sc); o[3] = __fdiv_rn(b.w, sc);
        for (int q = 0; q < 5; ++q)
            dimo[(size_t)r * 5 * nc + 5 * j + q] =
                __fadd_rn(__fmul_rn(dim_orien[(size_t)r * 5 * nc + 5 * j + q], 0.5f), dmean[q]);
    }
    int kd = 0, ld = 0, rd = 0;
    float km = kpts_prob[(size_t)r * 4 * grid];
    for (int e = 1; e < 4 * grid; ++e) { float v = kpts_prob[(size_t)r * 4 * grid + e]; if (v > km) { km = v; kd = e; } }
    float lm = left_prob[(size_t)r * grid], rm = right_prob[(size_t)r * grid];
    for (int e = 1; e < grid; ++e) {
        float v = left_prob[(size_t)r * grid + e]; if (v > lm) { lm = v; ld = e; }
        v = right_prob[(size_t)r * grid + e]; if (v > rm) { rm = v; rd = e; }
    }
    const float g = (float)grid;
    const float width = __fadd_rn(__fsub_rn(bl.z, bl.x), 1.0f);
    const float ktype = __fdiv_rn((float)kd, g);
    const float kdelta = fmodf((float)kd, g);
    const float pk = __fadd_rn(__fdiv_rn(__fmul_rn(kdelta, width), g), bl.x);
    const float pl = __fadd_rn(__fdiv_rn(__fmul_rn((float)ld, width), g), bl.x);
    const float pr = __fadd_rn(__fdiv_rn(__fmul_rn((float)rd, width), g), bl.x);
    float* o = pkpts + (size_t)r * 5;
    o[0] = __fdiv_rn(pk, sc); o[1] = ktype; o[2] = km; o[3] = __fdiv_rn(pl, sc); o[4] = __fdiv_rn(pr, sc);
    if (record) {
        // the per-image detection record that is all-gathered across ranks (SURVEY 8e / 8f-2): one row per RoI,
        // [scores nc | boxes_left 4nc | boxes_right 4nc | dim_orien 5nc | kpts 5], emitted here instead of a torch.cat
        float* q = record + (size_t)r * rec_ld;
        for (int j = 0; j < nc; ++j) *q++ = cls_prob[(size_t)r * nc + j];
        for (int j = 0; j < 4 * nc; ++j) *q++ = pbl[(size_t)r * 4 * nc + j];
        for (int j = 0; j < 4 * nc; ++j) *q++ = pbr[(size_t)r * 4 * nc + j];
        for (int j = 0; j < 5 * nc; ++j) *q++ = dimo[(size_t)r * 5 * nc + j];
        for (int j = 0; j < 5; ++j) *q++ = o[j];
    }
}


// per-class detection NMS of test_net.py:233-259 in one CTA (R <= 512): threshold, rank sort by score
// (desc, index asc), bitmask NMS, survivor-to-survivor greedy scan; keep[] = RoI indices in kept order.
__global__ void __launch_bounds__(512)
class_nms_kernel(const float* __restrict__ scores, const float* __restrict__ boxes, int R, int nc, int cls,
                 float score_thresh, float nms_thresh, int* __restrict__ keep, int* __restrict__ num) {
    __shared__ unsigned long long keys[512];
    __shared__ float4 sbox[512];
    __shared__ unsigned long long mask[512][8];
    __shared__ int n_valid;
    const int t = threadIdx.x;
    if (t == 0) n_valid = 0;
    unsigned long long k = 0;
    if (t < R) {
        const float s = scores[(size_t)t * nc + cls];
        if (s > score_thresh) {
            unsigned int b = __float_as_uint(s);
            b = (b & 0x80000000u) ? ~b : (b | 0x80000000u);
            k = ((unsigned long long)b << 32) | (unsigned long long)(0xFFFFFFFFu - (unsigned)t);
        }
    }
    keys[t] = k;
    __syncthreads();
    if (k) atomicAdd(&n_valid, 1);
    {   // rank sort (keys unique; zeros = below threshold rank last): 512 broadcast compares per thread
        int rank = 0;
#pragma unroll 8
        for (int j = 0; j < 512; ++j) rank += keys[j] > k;
        __syncthreads();
        if (k) keys[rank] = k;
        __syncthreads();
    }
    const int n = n_valid;
    if (t < n) {
        const int idx = (int)(0xFFFFFFFFu - (unsigned)(keys[t] & 0xFFFFFFFFu));
        const float* bp = boxes + (size_t)idx * 4 * nc + 4 * cls;
        sbox[t] = make_float4(bp[0], bp[1], bp[2], bp[3]);
    }
    __syncthreads();
    const int words = (n + 63) >> 6;
    for (int item = t; item < n * words; item += 512) {      // one (row, 64-box word) pair per work item
        const int row = item / words, w = item - row * words;
        const float4 cur = sbox[row];
        unsigned long long bits = 0;
        const int j0 = w * 64, j1 = min(n, j0 + 64);
        for (int j = max(j0, row + 1); j < j1; ++j)
            if (sb_iou_gt(cur, sbox[j], nms_thresh)) bits |= 1ULL << (j - j0);
        mask[row][w] = bits;
    }
    __syncthreads();
    if (t == 0) {   // greedy scan jumping from survivor to survivor
        unsigned long long remv[8] = {0, 0, 0, 0, 0, 0, 0, 0};
        int cnt = 0;
        for (int w = 0; w < words; ++w) {
            const int cs = min(n - w * 64, 64);
            const unsigned long long valid = cs >= 64 ? ~0ULL : ((1ULL << cs) - 1ULL);
            unsigned long long avail = ~remv[w] & valid;
            while (avail) {
                const int b = __ffsll((long long)avail) - 1;
                const int i = w * 64 + b;
                keep[cnt++] = (int)(0xFFFFFFFFu - (unsigned)(keys[i] & 0xFFFFFFFFu));
                for (int w2 = w; w2 < words; ++w2) remv[w2] |= mask[i][w2];
                const unsigned long long above = b >= 63 ? 0ULL : (~0ULL << (b + 1));
                avail = ~remv[w] & valid & above;
            }
        }
        *num = cnt;
    }
}

// Input pipeline (SURVEY 8f-3): prep_im_for_blob (lib/model/utils/blob.py:44-64) + HWC->CHW (demo.py:124-128):
// uint8 BGR image -> fp32 (pixel - PIXEL_MEANS) -> cv2.resize(fx=fy=scale, INTER_LINEAR) -> [3,Ho,Wo].
// OpenCV's separable fp32 bilinear restated: source coordinate (d+0.5)/scale-0.5 and its fraction in fp64, the
// horizontal pass on the two source rows first, then the vertical pass, one rounding per multiply / add.
struct ResizeTap { int i0, i1; float w0, w1; };
__device__ __forceinline__ ResizeTap resize_tap(int d, int n_src, double inv) {
    const double x = ((double)d + 0.5) * inv - 0.5;
    int s = (int)floor(x);
    float f = (float)(x - (double)s);
    if (s < 0) { f = 0.f; s = 0; }
    if (s >= n_src - 1) { f = 0.f; s = n_src - 1; }
    ResizeTap t;
    t.i0 = s; t.i1 = min(s + 1, n_src - 1);
    t.w0 = __fsub_rn(1.0f, f); t.w1 = f;
    return t;
}

__global__ void __launch_bounds__(256)
prep_image_kernel(const uint8_t* __restrict__ img, int H, int W, double inv, int rgb, float* __restrict__ out,
                  int Ho, int Wo) {
    const int x = blockIdx.x * 256 + threadIdx.x, y = blockIdx.y;
    if (x >= Wo) return;
    const ResizeTap tx = resize_tap(x, W, inv), ty = resize_tap(y, H, inv);
    const double means[3] = {102.9801, 115.9465, 122.7717};        // cfg.PIXEL_MEANS (config.py:170), BGR
    const uint8_t* r0 = img + (size_t)ty.i0 * W * 3;
    const uint8_t* r1 = img + (size_t)ty.i1 * W * 3;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        const int cs = rgb ? 2 - c : c;                            // demo.py:106-107: rgb -> bgr
        const float p00 = (float)((double)r0[tx.i0 * 3 + cs] - means[c]), p01 = (float)((double)r0[tx.i1 * 3 + cs] - means[c]);
        const float p10 = (float)((double)r1[tx.i0 * 3 + cs] - means[c]), p11 = (float)((double)r1[tx.i1 * 3 + cs] - means[c]);
        const float h0 = __fadd_rn(__fmul_rn(p00, tx.w0), __fmul_rn(p01, tx.w1));
        const float h1 = __fadd_rn(__fmul_rn(p10, tx.w0), __fmul_rn(p11, tx.w1));
        out[((size_t)c * Ho + y) * Wo + x] = __fadd_rn(__fmul_rn(h0, ty.w0), __fmul_rn(h1, ty.w1));
    }
}

}  // namespace

extern "C" int sb_prep_image_size(int H, int W, double scale, int* Ho, int* Wo) {
    if (!Ho || !Wo || H < 1 || W < 1 || !(scale > 0)) return SB_EINVAL;
    *Ho = (int)rint((double)H * scale);        // cv::saturate_cast<int>(ssize * inv_scale): round half to even
    *Wo = (int)rint((double)W * scale);
    return SB_OK;
}

extern "C" int sb_prep_image(const uint8_t* img, int H, int W, double scale, int rgb_input, float* out,
                             sb_stream_t stream) {
    int Ho = 0, Wo = 0;
    if (!img || !out || sb_prep_image_size(H, W, scale, &Ho, &Wo) != SB_OK || Ho < 1 || Wo < 1) return SB_EINVAL;
    prep_image_kernel<<<dim3(sb_div_up(Wo, 256), Ho), 256, 0, sb_cs(stream)>>>(img, H, W, 1.0 / scale, rgb_input, out, Ho, Wo);
    SB_LAUNCHED();
    SB_CHECK_LAUNCH();
    return SB_OK;
}

extern "C" int sb_fill(float* p, size_t n, float v, sb_stream_t stream) {
    if (n == 0) return SB_OK;
    if (n & 3) return SB_EINVAL;
    fill_kernel<<<148 * 8, 256, 0, sb_cs(stream)>>>((float4*)p, n / 4, v);
    SB_LAUNCHED();
    SB_CHECK_LAUNCH();
    return SB_OK;
}

extern "C" int sb_maxpool3x3s2_ceil(const float* in, int N, int H, int W, int C, float* out, sb_stream_t stream) {
    if (C & 3) return SB_EINVAL;
    auto osz = [](int x) { int o = (x - 3 + 1) / 2 + 1; if ((o - 1) * 2 >= x) --o; return o; };  // ceil mode
    const int Ho = osz(H), Wo = osz(W);
    const long long total = (long long)N * Ho * Wo * (C / 4);
    maxpool_kernel<<<sb_div_up(total, 256), 256, 0, sb_cs(stream)>>>((const float4*)in, N, H, W, C / 4, Ho, Wo, (float4*)out);
    SB_LAUNCHED();
    SB_CHECK_LAUNCH();
    return SB_OK;
}

extern "C" int sb_maxpool3x3s2_ceil16(const void* in, int N, int H, int W, int C, void* out, sb_stream_t stream) {
    if (C & 7) return SB_EINVAL;
    auto osz = [](int x) { int o = (x - 3 + 1) / 2 + 1; if ((o - 1) * 2 >= x) --o; return o; };
    const int Ho = osz(H), Wo = osz(W);
    const long long total = (long long)N * Ho * Wo * (C / 8);
    maxpool16_kernel<<<sb_div_up(total, 256), 256, 0, sb_cs(stream)>>>((const uint4*)in, N, H, W, C / 8, Ho, Wo, (uint4*)out);
    SB_LAUNCHED();
    SB_CHECK_LAUNCH();
    return SB_OK;
}

extern "C" int sb_subsample2(const float* in, int N, int H, int W, int C, float* out, sb_stream_t stream) {
    if (C & 3) return SB_EINVAL;
    const int Ho = (H - 1) / 2 + 1, Wo = (W - 1) / 2 + 1;
    const long long total = (long long)N * Ho * Wo * (C / 4);
    subsample2_kernel<<<sb_div_up(total, 256), 256, 0, sb_cs(stream)>>>((const float4*)in, N, H, W, C / 4, Ho, Wo, (float4*)out);
    SB_LAUNCHED();
    SB_CHECK_LAUNCH();
    return SB_OK;
}

extern "C" int sb_kpts_tail(const void* x, int x_is_half, int R, int G, int C, const float* w, const float* b,
                            float* kpts_prob, float* left_prob, float* right_prob, float* kpts_pred_all,
                            sb_stream_t stream) {
    if (R == 0) return SB_OK;
    if (!kpts_pred_all) return SB_EINVAL;     // [R,6,G] logits are also the staging buffer between the two kernels
    const int groups = 4, cols = (G + groups - 1) / groups;
    if (x_is_half && C == 256)
        kpts_colsum16_kernel<<<dim3(R, (G + 7) / 8), 256, 0, sb_cs(stream)>>>((const __half*)x, G, C, w, b, kpts_pred_all);
    else if (x_is_half)
        kpts_colsum_kernel<__half><<<dim3(R, groups), 256, 0, sb_cs(stream)>>>((const __half*)x, G, C, cols, w, b, kpts_pred_all);
    else
        kpts_colsum_kernel<float><<<dim3(R, groups), 256, 0, sb_cs(stream)>>>((const float*)x, G, C, cols, w, b, kpts_pred_all);
    SB_LAUNCHED();
    SB_CHECK_LAUNCH();
    kpts_softmax_kernel<<<R, 96, 0, sb_cs(stream)>>>(kpts_pred_all, G, kpts_prob, left_prob, right_prob);
    SB_LAUNCHED();
    SB_CHECK_LAUNCH();
    return SB_OK;
}

extern "C" int sb_box_tail(const float* fc7, int R, int K, int n_classes, const float* w_cls, const float* b_cls,
                           const float* w_box, const float* b_box, const float* w_dim, const float* b_dim,
                           float* cls_prob, float* bbox_pred, float* dim_orien, sb_stream_t stream) {
    if (R == 0) return SB_OK;
    if (n_classes < 1 || n_classes > 4) return SB_EINVAL;
    box_tail_kernel<false><<<R, 256, 0, sb_cs(stream)>>>(fc7, K, n_classes, w_cls, b_cls, w_box, b_box, w_dim, b_dim,
                                                         cls_prob, bbox_pred, dim_orien);
    SB_LAUNCHED();
    SB_CHECK_LAUNCH();
    return SB_OK;
}

extern "C" int sb_box_tail_logits(const float* fc7, int R, int K, int n_classes, const float* w_cls, const float* b_cls,
                                  const float* w_box, const float* b_box, const float* w_dim, const float* b_dim,
                                  float* cls_score, float* bbox_pred, float* dim_orien, sb_stream_t stream) {
    if (R == 0) return SB_OK;
    if (n_classes < 1 || n_classes > 4) return SB_EINVAL;
    box_tail_kernel<true><<<R, 256, 0, sb_cs(stream)>>>(fc7, K, n_classes, w_cls, b_cls, w_box, b_box, w_dim, b_dim,
                                                        cls_score, bbox_pred, dim_orien);
    SB_LAUNCHED();
    SB_CHECK_LAUNCH();
    return SB_OK;
}

extern "C" int sb_test_decode(const float* rois_left, const float* rois_right, const float* bbox_pred,
                              const float* dim_orien, const float* kpts_prob, const float* left_prob,
                              const float* right_prob, const float* im_info, int R, int n_classes, int grid,
                              float* pred_boxes_left, float* pred_boxes_right, float* dim_orien_out,
                              float* pred_kpts, sb_stream_t stream) {
    if (R == 0) return SB_OK;
    test_decode_kernel<<<sb_div_up(R, 128), 128, 0, sb_cs(stream)>>>(rois_left, rois_right, bbox_pred, dim_orien,
                                                                     kpts_prob, left_prob, right_prob, im_info, R,
                                                                     n_classes, grid, pred_boxes_left,
                                                                     pred_boxes_right, dim_orien_out, pred_kpts,
                                                                     nullptr, nullptr, 0);
    SB_LAUNCHED();
    SB_CHECK_LAUNCH();
    return SB_OK;
}

extern "C" int sb_test_decode_record(const float* rois_left, const float* rois_right, const float* cls_prob,
                                     const float* bbox_pred, const float* dim_orien, const float* kpts_prob,
                                     const float* left_prob, const float* right_prob, const float* im_info, int R,
                                     int n_classes, int grid, float* pred_boxes_left, float* pred_boxes_right,
                                     float* dim_orien_out, float* pred_kpts, float* record, int record_ld,
                                     sb_stream_t stream) {
    if (R == 0) return SB_OK;
    if (!cls_prob || !record || record_ld < 14 * n_classes + 5) return SB_EINVAL;
    test_decode_kernel<<<sb_div_up(R, 128), 128, 0, sb_cs(stream)>>>(rois_left, rois_right, bbox_pred, dim_orien,
                                                                     kpts_prob, left_prob, right_prob, im_info, R,
                                                                     n_classes, grid, pred_boxes_left,
                                                                     pred_boxes_right, dim_orien_out, pred_kpts,
                                                                     cls_prob, record, record_ld);
    SB_LAUNCHED();
    SB_CHECK_LAUNCH();
    return SB_OK;
}

extern "C" int sb_class_nms(const float* scores, const float* boxes, int R, int n_classes, int cls,
                            float score_thresh, float nms_thresh, int* keep, int* num_out, sb_stream_t stream) {
    if (R < 0 || R > 512 || cls < 0 || cls >= n_classes || !keep || !num_out) return SB_EINVAL;
    class_nms_kernel<<<1, 512, 0, sb_cs(stream)>>>(scores, boxes, R, n_classes, cls, score_thresh, nms_thresh, keep, num_out);
    SB_LAUNCHED();
    SB_CHECK_LAUNCH();
    return SB_OK;
}
