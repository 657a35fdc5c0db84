// Detect head decode: DFL softmax-expectation + anchor/dist2bbox + stride scale + class sigmoid in one pass
// (head.py:95-126, block.py:51-69, tal.py:326-350).  Input: per-level raw maps NHWC f32 with 4*reg_max box
// bins followed by nc class logits.  Output: (B, 4+nc, A) fp32, anchors level-major / row-major, or anchors
// [anchor_base, anchor_base + A) of a wider (B, 4+nc, y_anchors) prediction (one member of a model ensemble).
// A CTA takes 32 consecutive anchors of one image and level: the [32][no] tile is read with 16-B vectors
// (contiguous in NHWC), transposed through padded shared memory, and every output channel row is written as
// one 128-B coalesced segment.
#include "common.cuh"

namespace yl {

constexpr int kMaxLevels = 4;
struct DecodeParams {
    const float* x[kMaxLevels];
    long long cstride[kMaxLevels];
    int coff[kMaxLevels];
    int H[kMaxLevels], W[kMaxLevels];
    int tile0[kMaxLevels + 1];   // first tile index of each level
    int anchor0[kMaxLevels];     // first anchor of each level
    float stride[kMaxLevels];
    int nl, reg_max, nc, A;
    float* y;
};

__global__ void __launch_bounds__(256) detect_decode_kernel(const DecodeParams p) {
    extern __shared__ float tile[];  // [32][no + 1]
    __shared__ float dist[4][32];
    griddep_launch_dependents();
    griddep_wait();
    const int b = blockIdx.y;
    int lvl = 0;
    while (lvl + 1 < p.nl && (int)blockIdx.x >= p.tile0[lvl + 1]) ++lvl;
    const int HW = p.H[lvl] * p.W[lvl];
    const int a0 = ((int)blockIdx.x - p.tile0[lvl]) * 32;
    const int cnt = min(32, HW - a0);
    const int nbox = 4 * p.reg_max;
    const int no = nbox + p.nc;
    const int ld = no + 1;

    // ---- load [cnt][no]: 16-B vectors when no, coff and cstride are multiples of 4 (checked on the host), else
    // scalars (heads whose nc is not a multiple of 4)
    const float* src = p.x[lvl] + ((long long)b * HW + a0) * p.cstride[lvl] + p.coff[lvl];
    if ((no & 3) == 0) {
        const int v4 = no >> 2;
        for (int i = threadIdx.x; i < cnt * v4; i += blockDim.x) {
            const int px = i / v4, q = i - px * v4;
            const float4 t = __ldg(reinterpret_cast<const float4*>(src + (long long)px * p.cstride[lvl] + q * 4));
            float* d = tile + px * ld + q * 4;
            d[0] = t.x; d[1] = t.y; d[2] = t.z; d[3] = t.w;
        }
    } else {
        for (int i = threadIdx.x; i < cnt * no; i += blockDim.x) {
            const int px = i / no, q = i - px * no;
            tile[px * ld + q] = __ldg(src + (long long)px * p.cstride[lvl] + q);
        }
    }
    __syncthreads();

    // ---- DFL: thread (side, px) -> expected bin
    if (threadIdx.x < 128) {
        const int side = threadIdx.x >> 5, px = threadIdx.x & 31;
        float e = 0.f;
        if (px < cnt) {
            const float* l = tile + px * ld + side * p.reg_max;
            float m = l[0];
            for (int k = 1; k < p.reg_max; ++k) m = fmaxf(m, l[k]);
            float s = 0.f;
            for (int k = 0; k < p.reg_max; ++k) {
                const float w = expf(l[k] - m);
                s += w;
                e += w * (float)k;
            }
            e /= s;
        }
        dist[side][px] = e;
    }
    __syncthreads();
    float* yb = p.y + (long long)b * (4 + p.nc) * p.A + p.anchor0[lvl] + a0;
    if (threadIdx.x < 128) {
        const int ch = threadIdx.x >> 5, px = threadIdx.x & 31;
        if (px < cnt) {
            const int a = a0 + px;
            const float ax = (float)(a % p.W[lvl]) + 0.5f, ay = (float)(a / p.W[lvl]) + 0.5f;
            const float x1 = ax - dist[0][px], y1 = ay - dist[1][px];
            const float x2 = ax + dist[2][px], y2 = ay + dist[3][px];
            float v;
            if (ch == 0) v = (x1 + x2) / 2.f;
            else if (ch == 1) v = (y1 + y2) / 2.f;
            else if (ch == 2) v = x2 - x1;
            else v = y2 - y1;
            yb[(long long)ch * p.A + px] = v * p.stride[lvl];
        }
    }
    // ---- class scores
    for (int i = threadIdx.x; i < p.nc * 32; i += blockDim.x) {
        const int c = i >> 5, px = i & 31;
        if (px < cnt) {
            const float l = tile[px * ld + nbox + c];
            yb[(long long)(4 + c) * p.A + px] = 1.f / (1.f + expf(-l));
        }
    }
}

// Standalone DFL (block.py:51-69): x (b, 4*reg_max, a) fp32 channel-major -> (b, 4, a).
__global__ void __launch_bounds__(256) dfl_kernel(const float* __restrict__ x, float* __restrict__ y, int reg_max,
                                                  int a, long long total) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const int ai = (int)(i % a);
    const long long bs = i / a;  // b * 4 + side
    const float* l = x + bs * reg_max * a + ai;
    float m = l[0];
    for (int k = 1; k < reg_max; ++k) m = fmaxf(m, l[(long long)k * a]);
    float s = 0.f, e = 0.f;
    for (int k = 0; k < reg_max; ++k) {
        const float w = expf(l[(long long)k * a] - m);
        s += w;
        e += w * (float)k;
    }
    y[i] = e / s;
}

}  // namespace yl

extern "C" int yl_dfl(const float* x, float* y, int b, int reg_max, int a, void* stream) {
    YL_CHECK(x && y && b > 0 && reg_max > 0 && a > 0, YL_ERR_ARG, "bad arguments");
    const long long total = (long long)b * 4 * a;
    yl::dfl_kernel<<<(unsigned)yl::ceil_div64(total, 256), 256, 0, (cudaStream_t)stream>>>(x, y, reg_max, a, total);
    YL_LAUNCH_OK("dfl_kernel");
    return YL_OK;
}

extern "C" int yl_detect_decode_into(const yl_tensor* levels, int nl, const float* strides_host, int reg_max, int nc,
                                     float* y, int y_anchors, int anchor_base, void* stream) {
    YL_CHECK(levels && strides_host && y, YL_ERR_ARG, "null pointer");
    YL_CHECK(nl >= 1 && nl <= yl::kMaxLevels, YL_ERR_ARG, "1..%d levels supported", yl::kMaxLevels);
    YL_CHECK(reg_max >= 1 && nc >= 1, YL_ERR_ARG, "bad reg_max/nc");
    const int no = 4 * reg_max + nc;
    yl::DecodeParams p;
    int tiles = 0, A = 0;
    for (int i = 0; i < nl; ++i) {
        const yl_tensor& t = levels[i];
        YL_CHECK(t.data && t.dtype == YL_F32, YL_ERR_ARG, "level %d must be f32", i);
        YL_CHECK(t.c == no && t.coff + t.c <= t.cstride && (no % 4 || (t.coff % 4 == 0 && t.cstride % 4 == 0)),
                 YL_ERR_ARG, "level %d: channels %d (expected %d) / alignment", i, t.c, no);
        YL_CHECK(t.n == levels[0].n, YL_ERR_ARG, "batch mismatch at level %d", i);
        p.x[i] = reinterpret_cast<const float*>(t.data);
        p.cstride[i] = t.cstride;
        p.coff[i] = t.coff;
        p.H[i] = t.h;
        p.W[i] = t.w;
        p.tile0[i] = tiles;
        p.anchor0[i] = anchor_base + A;
        p.stride[i] = strides_host[i];
        tiles += yl::ceil_div(t.h * t.w, 32);
        A += t.h * t.w;
    }
    YL_CHECK(anchor_base >= 0 && y_anchors >= 0 && (long long)anchor_base + A <= y_anchors, YL_ERR_ARG,
             "anchor window [%d, %lld) outside the %d anchors of y", anchor_base, (long long)anchor_base + A, y_anchors);
    p.tile0[nl] = tiles;
    p.nl = nl;
    p.reg_max = reg_max;
    p.nc = nc;
    p.A = y_anchors;
    p.y = y;
    const size_t smem = (size_t)32 * (no + 1) * sizeof(float);
    YL_CHECK(smem <= 48 * 1024, YL_ERR_UNSUPPORTED, "too many head channels (%d)", no);
    dim3 grid((unsigned)tiles, (unsigned)levels[0].n, 1);
    YL_CUDA(yl::launch_kernel(yl::detect_decode_kernel, grid, dim3(256), smem, (cudaStream_t)stream, p));
    YL_LAUNCH_OK("detect_decode_kernel");
    return YL_OK;
}

extern "C" int yl_detect_decode(const yl_tensor* levels, int nl, const float* strides_host, int reg_max, int nc,
                                float* y, void* stream) {
    YL_CHECK(levels && nl >= 1 && nl <= yl::kMaxLevels, YL_ERR_ARG, "1..%d levels supported", yl::kMaxLevels);
    int A = 0;
    for (int i = 0; i < nl; ++i) A += levels[i].h * levels[i].w;
    return yl_detect_decode_into(levels, nl, strides_host, reg_max, nc, y, A, 0, stream);
}
