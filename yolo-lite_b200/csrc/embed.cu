// Feature embeddings (BaseModel._predict_once with `embed`, nn/tasks.py): adaptive_avg_pool2d(x, (1, 1)) of every tapped
// layer output, concatenated along channels into one (B, D) fp32 matrix, all taps in ONE launch.
//
// Work item = (tap, image, group tile, pixel chunk): a block of 256 threads covers up to 256 8-channel groups of one
// image and a fixed range of pixels; each thread reads 16 B (8 bf16 channels) per pixel and keeps 8 fp32 sums.  The
// pixel split gives every tap size enough blocks to stream at HBM rate (a 160x160x64 tap at bs 64 is only 64
// image x group-tile pairs).  The partition is a pure function of (h*w, c), so the result is deterministic and the same
// for an image whatever batch it is in: the lanes of a block are combined in lane order, and the chunk partials of an
// item go to a workspace slot each; the block that finishes an item last (an integer counter per item) adds them in
// chunk order, writes the mean and resets the counter, so the workspace is all zeros again after every launch.
#include "common.cuh"

namespace yl {

constexpr int kEmbedThreads = 256;
constexpr int kEmbedMaxTaps = 32;
constexpr int kEmbedChunkBytes = 64 << 10;   // bytes one block reads per pixel chunk (16 loads per thread at 8 groups)

struct EmbedTapParams {
    const __nv_bfloat16* x;  // channel `coff` of pixel 0 of image 0
    long long cstride;
    long long ws0;           // first partial (float) of this tap in the workspace (nchunk > 1)
    long long cnt0;          // first item counter of this tap (nchunk > 1)
    int hw, G;               // pixels per image, 8-channel groups
    int gtiles, nchunk, ppc; // group tiles of <= 256 groups, pixel chunks per item, pixels per chunk
    int col;                 // first output column
    int block0;              // first block of this tap
    float inv_hw;
};

struct EmbedParams {
    EmbedTapParams t[kEmbedMaxTaps];
    int n_taps, D;
    float* out;
    float* ws;
    unsigned* cnt;
};

__device__ __forceinline__ void add_bf16x8(float (&acc)[8], const uint4 v) {
    const uint32_t u[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        acc[2 * k] += __uint_as_float(u[k] << 16);
        acc[2 * k + 1] += __uint_as_float(u[k] & 0xffff0000u);
    }
}

__global__ void __launch_bounds__(kEmbedThreads) embed_pool_kernel(const __grid_constant__ EmbedParams p) {
    __shared__ float red[kEmbedThreads * 8];
    __shared__ int s_last;
    griddep_launch_dependents();
    griddep_wait();
    int b = blockIdx.x, ti = 0;
    while (ti + 1 < p.n_taps && b >= p.t[ti + 1].block0) ++ti;
    const EmbedTapParams& T = p.t[ti];
    b -= T.block0;
    const int chunk = b % T.nchunk;
    b /= T.nchunk;
    const int gt = b % T.gtiles, n = b / T.gtiles;
    const int g0 = gt * kEmbedThreads;
    const int Gb = min(T.G - g0, kEmbedThreads);      // groups of this tile
    const int P = kEmbedThreads / Gb;                 // pixel lanes
    const int lane = threadIdx.x / Gb, g = threadIdx.x - lane * Gb;
    float acc[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) acc[k] = 0.f;
    if (lane < P) {
        const int p1 = min((chunk + 1) * T.ppc, T.hw);
        const __nv_bfloat16* src = T.x + (long long)n * T.hw * T.cstride + (g0 + g) * 8;
        int px = chunk * T.ppc + lane;
        for (; px + 3 * P < p1; px += 4 * P) {   // four loads in flight per thread
            uint4 v[4];
#pragma unroll
            for (int k = 0; k < 4; ++k)
                v[k] = __ldcs(reinterpret_cast<const uint4*>(src + (long long)(px + k * P) * T.cstride));
#pragma unroll
            for (int k = 0; k < 4; ++k) add_bf16x8(acc, v[k]);
        }
        for (; px < p1; px += P) add_bf16x8(acc, __ldcs(reinterpret_cast<const uint4*>(src + (long long)px * T.cstride)));
#pragma unroll
        for (int k = 0; k < 8; ++k) red[(lane * Gb + g) * 8 + k] = acc[k];
    }
    __syncthreads();
    const int E = Gb * 8;                            // output columns of this item
    float* out = p.out + (long long)n * p.D + T.col + g0 * 8;
    if (T.nchunk == 1) {
        for (int e = threadIdx.x; e < E; e += kEmbedThreads) {
            float s = 0.f;
            for (int l = 0; l < P; ++l) s += red[l * E + e];
            out[e] = s * T.inv_hw;
        }
        return;
    }
    const long long item = (long long)n * T.gtiles + gt;
    const int S = min(T.G, kEmbedThreads) * 8;       // partial slot stride (the widest tile)
    float* part = p.ws + T.ws0 + item * T.nchunk * S;
    for (int e = threadIdx.x; e < E; e += kEmbedThreads) {
        float s = 0.f;
        for (int l = 0; l < P; ++l) s += red[l * E + e];
        __stcg(part + (long long)chunk * S + e, s);
    }
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) s_last = atomicAdd(p.cnt + T.cnt0 + item, 1u) == (unsigned)(T.nchunk - 1);
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    for (int e = threadIdx.x; e < E; e += kEmbedThreads) {
        float s = 0.f;
        for (int k = 0; k < T.nchunk; ++k) s += __ldcg(part + (long long)k * S + e);
        out[e] = s * T.inv_hw;
    }
    if (threadIdx.x == 0) p.cnt[T.cnt0 + item] = 0u;   // ready for the next launch (graph replay)
}

}  // namespace yl

extern "C" int yl_embed_pool(const yl_embed_tap* taps, int n_taps, int B, int D, float* out, void* workspace,
                             size_t* workspace_bytes, void* stream) {
    YL_CHECK(taps && workspace_bytes, YL_ERR_ARG, "null pointer");
    YL_CHECK(n_taps >= 1 && n_taps <= yl::kEmbedMaxTaps, YL_ERR_ARG, "embed_pool takes 1..%d taps (got %d)",
             yl::kEmbedMaxTaps, n_taps);
    YL_CHECK(B >= 1 && D >= 1, YL_ERR_ARG, "bad embed_pool output (%d, %d)", B, D);
    yl::EmbedParams p;
    long long blocks = 0, ws_floats = 0, counters = 0;
    for (int i = 0; i < n_taps; ++i) {
        const yl_tensor& x = taps[i].x;
        YL_CHECK(x.data && ((uintptr_t)x.data % 16) == 0 && x.dtype == YL_BF16, YL_ERR_ARG,
                 "tap %d: null, not 16-byte aligned or not bf16", i);
        YL_CHECK(x.n == B && x.h >= 1 && x.w >= 1 && x.c >= 8, YL_ERR_ARG, "tap %d: bad dims (%d, %d, %d, %d) for B %d", i,
                 x.n, x.h, x.w, x.c, B);
        YL_CHECK(x.c % 8 == 0 && x.coff % 8 == 0 && x.cstride % 8 == 0 && x.coff >= 0 && x.coff + x.c <= x.cstride,
                 YL_ERR_ARG, "tap %d: c %d, coff %d and cstride %d must be multiples of 8 with coff + c <= cstride", i, x.c,
                 x.coff, x.cstride);
        YL_CHECK(taps[i].col >= 0 && taps[i].col + x.c <= D, YL_ERR_ARG, "tap %d: columns [%d, %d) outside D %d", i,
                 taps[i].col, taps[i].col + x.c, D);
        yl::EmbedTapParams& t = p.t[i];
        t.x = reinterpret_cast<const __nv_bfloat16*>(x.data) + x.coff;
        t.cstride = x.cstride;
        t.hw = x.h * x.w;
        t.G = x.c / 8;
        t.gtiles = yl::ceil_div(t.G, yl::kEmbedThreads);
        const int Gb = t.G < yl::kEmbedThreads ? t.G : yl::kEmbedThreads;
        const int P = yl::kEmbedThreads / Gb;
        int ppc = yl::kEmbedChunkBytes / (Gb * 16);
        ppc = yl::ceil_div(ppc < 1 ? 1 : ppc, P) * P;          // every pixel lane gets the same number of pixels
        t.ppc = ppc < t.hw ? ppc : t.hw;
        t.nchunk = yl::ceil_div(t.hw, t.ppc);
        t.col = taps[i].col;
        t.inv_hw = 1.0f / (float)t.hw;
        const long long items = (long long)B * t.gtiles;
        t.block0 = (int)blocks;
        blocks += items * t.nchunk;
        YL_CHECK(blocks < (1ll << 31), YL_ERR_ARG, "embed_pool grid too large");
        t.ws0 = ws_floats;
        t.cnt0 = counters;
        if (t.nchunk > 1) {
            ws_floats += items * t.nchunk * Gb * 8;
            counters += items;
        }
    }
    const size_t cnt_off = ((size_t)ws_floats * sizeof(float) + 15) / 16 * 16;
    const size_t need = cnt_off + (size_t)counters * sizeof(unsigned);
    if (!workspace) {
        *workspace_bytes = need;
        return YL_OK;
    }
    YL_CHECK(out && ((uintptr_t)workspace % 16) == 0, YL_ERR_ARG, "null output or unaligned workspace");
    YL_CHECK(*workspace_bytes >= need, YL_ERR_WORKSPACE, "embed_pool workspace %zu B < %zu B", *workspace_bytes, need);
    p.n_taps = n_taps;
    p.D = D;
    p.out = out;
    p.ws = reinterpret_cast<float*>(workspace);
    p.cnt = reinterpret_cast<unsigned*>(reinterpret_cast<char*>(workspace) + cnt_off);
    YL_CUDA(yl::launch_kernel(yl::embed_pool_kernel, dim3((unsigned)blocks), dim3(yl::kEmbedThreads), 0,
                              (cudaStream_t)stream, p));
    YL_LAUNCH_OK("embed_pool_kernel");
    return YL_OK;
}
