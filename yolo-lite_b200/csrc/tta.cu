// Test-time augmentation (DetectionModel._predict_augment, nn/tasks.py): the two elementwise steps around the three
// model passes.
//
//   yl_tta_scale_img: scale_img (utils/torch_utils.py) of the flipped / unflipped input for passes 1 and 2 in ONE launch.
//     A block owns a band of input rows of one (image, channel) plane: it stages them in shared memory as fp32 (widening
//     fp16, dividing uint8 by 255) with 16-byte loads, then writes every output row of BOTH canvases whose top source
//     row lies in the band, as float4 stores; a thread keeps the horizontal taps of its 4 output columns in registers
//     for all rows.  Each input row is therefore fetched from HBM once for both passes (plus
//     the one boundary row a band shares with the next).
//     Arithmetic is PyTorch's upsample_bilinear2d (align_corners=False, size given): scale = (float)in / out,
//     src = max(scale * (dst + 0.5) - 0.5, 0), i0 = (int)src, i0 + 1 clamped, lambda1 = src - i0.  The expressions are
//     written as ATen's kernel writes them and this file is compiled without fast-math, so nvcc contracts them the same
//     way.  Pixels right of / below the content get F.pad's 0.447.
//
//   yl_tta_merge: _descale_pred + _clip_augmented + torch.cat(y, -1).  Bit-identical to torch on the GPU: the box rows
//     are multiplied by the fp32 reciprocal of the scale (what `p[:, :4] /= scale` does for a Python scalar on CUDA),
//     and the flipped pass's x is `img_w - x`, each rounded separately (explicit _rn intrinsics: no FMA contraction).
#include "common.cuh"

#include <cuda_fp16.h>

namespace yl {

constexpr int kTtaThreads = 256;
constexpr int kTtaSmemBytes = 48 * 1024;   // most shared memory a block stages (no opt-in needed) ...
constexpr int kTtaBandBytes = 32 * 1024;   // ... and the band it aims for: ~7 blocks of 256 threads per SM
constexpr float kTtaPad = 0.447f;          // scale_img's F.pad value

struct TtaScaleParams {
    const void* x;
    int dtype, c, h, w;
    int band;          // input rows per block
    int vec;           // 16-byte loads are aligned
    yl_tta_canvas cv[2];
    float sh[2], sw[2];   // (float)in / out per axis
};

// top source row / column of destination index d (area_pixel_compute_source_index, cubic = false)
__device__ __forceinline__ float tta_src(float scale, int d) {
    const float s = scale * ((float)d + 0.5f) - 0.5f;
    return s < 0.f ? 0.f : s;
}
__device__ __forceinline__ int tta_i0(float scale, int d) { return (int)tta_src(scale, d); }

template <int DT>
__device__ __forceinline__ float tta_load1(const void* x, long long i) {
    if (DT == YL_F32) return __ldg(reinterpret_cast<const float*>(x) + i);
    if (DT == YL_F16) return __half2float(reinterpret_cast<const __half*>(x)[i]);
    return __fdiv_rn((float)__ldg(reinterpret_cast<const uint8_t*>(x) + i), 255.f);   // true division, like yl_to_f32
}

// one 16-byte load of DT elements -> fp32 in smem
template <int DT>
__device__ __forceinline__ void tta_widen16(const uint4 q, float* o) {
    if (DT == YL_F32) {
        *reinterpret_cast<float4*>(o) = make_float4(__uint_as_float(q.x), __uint_as_float(q.y), __uint_as_float(q.z),
                                                    __uint_as_float(q.w));
    } else if (DT == YL_F16) {
        const uint32_t wd[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
        for (int k = 0; k < 8; ++k) o[k] = __half2float(__ushort_as_half((unsigned short)(wd[k >> 1] >> (16 * (k & 1)))));
    } else {
        const uint32_t wd[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
        for (int k = 0; k < 16; ++k) o[k] = __fdiv_rn((float)((wd[k >> 2] >> (8 * (k & 3))) & 0xffu), 255.f);
    }
}

// n consecutive elements starting at element `base` -> smem fp32.  Four 16-byte loads per thread are issued before
// their results are used: with one load in flight per thread the staging phase is latency-bound, not HBM-bound.
template <int DT>
__device__ __forceinline__ void tta_stage(const void* x, long long base, int n, bool vec, float* s) {
    constexpr int E = DT == YL_F32 ? 4 : (DT == YL_F16 ? 8 : 16);   // elements per 16-byte load
    constexpr int U = 4;
    if (vec) {
        const uint4* src = reinterpret_cast<const uint4*>(reinterpret_cast<const char*>(x) + base * (16 / E));
        const int nv = n / E;
        int v = threadIdx.x;
        for (; v + (U - 1) * kTtaThreads < nv; v += U * kTtaThreads) {
            uint4 q[U];
#pragma unroll
            for (int u = 0; u < U; ++u) q[u] = __ldg(src + v + u * kTtaThreads);
#pragma unroll
            for (int u = 0; u < U; ++u) tta_widen16<DT>(q[u], s + (v + u * kTtaThreads) * E);
        }
        for (; v < nv; v += kTtaThreads) tta_widen16<DT>(__ldg(src + v), s + v * E);
        for (int i = nv * E + threadIdx.x; i < n; i += kTtaThreads) s[i] = tta_load1<DT>(x, base + i);
    } else {
        for (int i = threadIdx.x; i < n; i += kTtaThreads) s[i] = tta_load1<DT>(x, base + i);
    }
}

template <int DT>
__global__ void __launch_bounds__(kTtaThreads) tta_scale_img_kernel(const TtaScaleParams p) {
    extern __shared__ float rows[];   // staged input rows [a, a + nrows) of this plane, fp32
    const int plane = blockIdx.y;     // image * c + channel
    const int a = blockIdx.x * p.band;
    const int b = min(a + p.band, p.h);            // this block owns output rows whose top source row is in [a, b)
    const int last = min(b, p.h - 1);              // ... and reads rows [a, last] (i0 + 1 is clamped)
    const int nrows = last - a + 1;
    tta_stage<DT>(p.x, ((long long)plane * p.h + a) * p.w, nrows * p.w, p.vec != 0, rows);
    __syncthreads();
    const bool last_band = b == p.h;
    // output rows [y0, y1) of each canvas: the content rows whose top source row i0(y) (non-decreasing in y) is in [a, b)
    int y0[2], y1[2];
#pragma unroll   // constant k: the parameter arrays are indexed statically (no local-memory copy)
    for (int k = 0; k < 2; ++k) {
        const float sh = p.sh[k];
        int lo = max(0, (int)((float)a / sh) - 2);
        while (lo > 0 && tta_i0(sh, lo - 1) >= a) --lo;
        while (lo < p.cv[k].h && tta_i0(sh, lo) < a) ++lo;
        int hi = lo;
        while (hi < p.cv[k].h && tta_i0(sh, hi) < b) ++hi;
        y0[k] = lo;
        y1[k] = last_band ? p.cv[k].H : hi;   // the last band also writes the pad rows below the content
    }
    // a thread owns groups of 4 output columns of one canvas (the column groups of both canvases are numbered one after
    // the other): it computes their horizontal taps once and walks the band's rows with them
    const int q0 = p.cv[0].W >> 2, q1 = p.cv[1].W >> 2;
    for (int gi = threadIdx.x; gi < q0 + q1; gi += kTtaThreads) {
        const bool k0 = gi < q0;   // selects field by field: a reference to p.cv[k] would copy p to local memory
        float* const cy = k0 ? p.cv[0].y : p.cv[1].y;
        const int cH = k0 ? p.cv[0].H : p.cv[1].H, cW = k0 ? p.cv[0].W : p.cv[1].W;
        const int ch = k0 ? p.cv[0].h : p.cv[1].h, cw = k0 ? p.cv[0].w : p.cv[1].w;
        const int flip = k0 ? p.cv[0].flip : p.cv[1].flip;
        const float sh = k0 ? p.sh[0] : p.sh[1], sw = k0 ? p.sw[0] : p.sw[1];
        const int x0 = (gi - (k0 ? 0 : q0)) * 4;
        int c0[4], c1[4];
        float w0l[4], w1l[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const float wr = tta_src(sw, x0 + j);
            const int w1 = (int)wr;
            const int w1p = w1 < p.w - 1 ? 1 : 0;
            w1l[j] = wr - (float)w1;
            w0l[j] = 1.f - w1l[j];
            // flip before resize: column c of the flipped image is column w - 1 - c of the input
            c0[j] = flip ? p.w - 1 - w1 : w1;
            c1[j] = flip ? c0[j] - w1p : c0[j] + w1p;
            if (x0 + j >= cw) c0[j] = c1[j] = -1;   // pad column
        }
        const int ys = k0 ? y0[0] : y0[1], ye = k0 ? y1[0] : y1[1];
        float* out = cy + ((long long)plane * cH + ys) * cW + x0;
        for (int y = ys; y < ye; ++y, out += cW) {
            float v[4];
            if (y >= ch) {
                v[0] = v[1] = v[2] = v[3] = kTtaPad;
            } else {
                const float hr = tta_src(sh, y);
                const int h1 = (int)hr;
                const int h1p = h1 < p.h - 1 ? 1 : 0;
                const float h1l = hr - (float)h1;
                const float h0l = 1.f - h1l;
                const float* r0 = rows + (h1 - a) * p.w;
                const float* r1 = r0 + h1p * p.w;
#pragma unroll
                for (int j = 0; j < 4; ++j)
                    v[j] = c0[j] < 0 ? kTtaPad
                                     : h0l * (w0l[j] * r0[c0[j]] + w1l[j] * r0[c1[j]]) +
                                           h1l * (w0l[j] * r1[c0[j]] + w1l[j] * r1[c1[j]]);
            }
            *reinterpret_cast<float4*>(out) = make_float4(v[0], v[1], v[2], v[3]);
        }
    }
}

struct TtaMergeParams {
    const float* pred[3];
    int A[3], a0[3], n[3];
    float inv[3];      // fp32 reciprocal of the pass scale
    int flip[3];
    int rows, A_out;   // 4 + nc, sum of n
    float img_w;
};

constexpr int kMergePerThread = 8;

// a[s] for s in {0, 1, 2} without a dynamically indexed (local-memory) copy of the parameter array
template <typename T>
__device__ __forceinline__ T pick3(const T (&a)[3], int s) {
    return s == 0 ? a[0] : (s == 1 ? a[1] : a[2]);
}

// grid: (row chunks, (4 + nc) * B); each thread moves kMergePerThread elements of one output row, 4-byte accesses that
// are fully coalesced across the warp (rows of odd length rule out 16-byte alignment)
__global__ void __launch_bounds__(kTtaThreads) tta_merge_kernel(const TtaMergeParams p, float* __restrict__ y) {
    const int row = blockIdx.y;            // image * rows + r
    const int r = row % p.rows;
    const int img = row / p.rows;
    float* out = y + (long long)row * p.A_out;
    const int e0 = blockIdx.x * (kTtaThreads * kMergePerThread) + threadIdx.x;
    float v[kMergePerThread];
    int seg[kMergePerThread];
#pragma unroll
    for (int k = 0; k < kMergePerThread; ++k) {   // all loads first: kMergePerThread requests in flight per thread
        int e = e0 + k * kTtaThreads;
        seg[k] = 0;
        if (e >= p.A_out) continue;
        if (e >= p.n[0]) {
            e -= p.n[0];
            seg[k] = 1;
            if (e >= p.n[1]) {
                e -= p.n[1];
                seg[k] = 2;
            }
        }
        const int s = seg[k];
        v[k] = __ldg(pick3(p.pred, s) + ((long long)img * p.rows + r) * pick3(p.A, s) + pick3(p.a0, s) + e);
    }
#pragma unroll
    for (int k = 0; k < kMergePerThread; ++k) {
        const int e = e0 + k * kTtaThreads;
        if (e >= p.A_out) continue;
        float t = v[k];
        if (r < 4) {
            t = __fmul_rn(t, pick3(p.inv, seg[k]));                          // p[:, :4] /= scale
            if (r == 0 && pick3(p.flip, seg[k])) t = __fsub_rn(p.img_w, t);   // x = img_size[1] - x
        }
        out[e] = t;
    }
}

}  // namespace yl

extern "C" {

int yl_tta_scale_img(const void* x, int x_dtype, int n, int c, int h, int w, const yl_tta_canvas* canvases,
                     void* stream) {
    YL_CHECK(x && canvases, YL_ERR_ARG, "null pointer");
    YL_CHECK(x_dtype == YL_F32 || x_dtype == YL_F16 || x_dtype == YL_U8, YL_ERR_ARG,
             "tta_scale_img reads YL_F32, YL_F16 or YL_U8 (got dtype %d)", x_dtype);
    YL_CHECK(n >= 1 && c >= 1 && (long long)n * c <= 65535 && h >= 1 && w >= 1, YL_ERR_ARG, "bad tta_scale_img input dims");
    yl::TtaScaleParams p;
    p.x = x;
    p.dtype = x_dtype;
    p.c = c;
    p.h = h;
    p.w = w;
    for (int k = 0; k < 2; ++k) {
        const yl_tta_canvas& cv = canvases[k];
        YL_CHECK(cv.y && ((uintptr_t)cv.y % 16) == 0, YL_ERR_ARG, "canvas %d: null or not 16-byte aligned", k);
        YL_CHECK(cv.h >= 1 && cv.w >= 1 && cv.h <= cv.H && cv.w <= cv.W && cv.W % 4 == 0, YL_ERR_ARG,
                 "canvas %d: content %dx%d must fit the canvas %dx%d (W %% 4 == 0)", k, cv.h, cv.w, cv.H, cv.W);
        p.cv[k] = cv;
        p.sh[k] = (float)h / (float)cv.h;
        p.sw[k] = (float)w / (float)cv.w;
    }
    const int row_bytes = (int)sizeof(float) * w;
    YL_CHECK(2 * row_bytes <= yl::kTtaSmemBytes, YL_ERR_UNSUPPORTED, "tta_scale_img stages at least two rows of %d pixels "
             "in 48 KB", w);
    p.band = min(max(yl::kTtaBandBytes / row_bytes, 2) - 1, h);
    const int esize = x_dtype == YL_F32 ? 4 : (x_dtype == YL_F16 ? 2 : 1);
    p.vec = ((uintptr_t)x % 16 == 0 && ((long long)w * esize) % 16 == 0) ? 1 : 0;
    const dim3 grid((unsigned)yl::ceil_div(h, p.band), (unsigned)(n * c)), block(yl::kTtaThreads);
    const size_t smem = sizeof(float) * (size_t)min(p.band + 1, h) * w;
    cudaStream_t s = (cudaStream_t)stream;
    if (x_dtype == YL_F32)
        yl::tta_scale_img_kernel<YL_F32><<<grid, block, smem, s>>>(p);
    else if (x_dtype == YL_F16)
        yl::tta_scale_img_kernel<YL_F16><<<grid, block, smem, s>>>(p);
    else
        yl::tta_scale_img_kernel<YL_U8><<<grid, block, smem, s>>>(p);
    YL_LAUNCH_OK("tta_scale_img_kernel");
    return YL_OK;
}

int yl_tta_merge(const yl_tta_pass* passes, int B, int nc, int img_w, float* y, void* stream) {
    YL_CHECK(passes && y, YL_ERR_ARG, "null pointer");
    YL_CHECK(B >= 1 && nc >= 1 && (long long)B * (4 + nc) <= 65535, YL_ERR_ARG, "bad tta_merge dims (B %d, nc %d)", B, nc);
    yl::TtaMergeParams p;
    long long total = 0;
    for (int k = 0; k < 3; ++k) {
        const yl_tta_pass& q = passes[k];
        YL_CHECK(q.pred && q.A >= 1 && q.a0 >= 0 && q.n >= 0 && q.a0 + q.n <= q.A && q.scale > 0.f, YL_ERR_ARG,
                 "pass %d: bad prediction or kept range [%d, %d) of %d anchors", k, q.a0, q.a0 + q.n, q.A);
        p.pred[k] = q.pred;
        p.A[k] = q.A;
        p.a0[k] = q.a0;
        p.n[k] = q.n;
        p.inv[k] = 1.0f / q.scale;   // torch: a * (1 / b) for a CPU-scalar divisor, computed in the op's fp32
        p.flip[k] = q.flip;
        total += q.n;
    }
    YL_CHECK(total >= 1 && total < (1ll << 31), YL_ERR_ARG, "bad merged anchor count %lld", total);
    p.rows = 4 + nc;
    p.A_out = (int)total;
    p.img_w = (float)img_w;
    const int per_block = yl::kTtaThreads * yl::kMergePerThread;
    const dim3 grid((unsigned)yl::ceil_div(p.A_out, per_block), (unsigned)(B * p.rows)), block(yl::kTtaThreads);
    yl::tta_merge_kernel<<<grid, block, 0, (cudaStream_t)stream>>>(p, y);
    YL_LAUNCH_OK("tta_merge_kernel");
    return YL_OK;
}

}  // extern "C"
