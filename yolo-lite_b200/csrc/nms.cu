// Batched non-max suppression on the GPU, bit-exact against the reference's CPU path
// (utils/ops.py:138-273 + torchvision.ops.nms CPU kernel).
//
// Kernel 1  nms_filter_kernel   HBM-bound sweep over the (B, 4+nc, A) prediction tensor, coalesced along the
//                               anchor axis (float4 per thread).  Confidence test (strict >), best class or
//                               multi-label expansion, optional class filter, warp-ballot aggregated
//                               compaction.  A candidate is one 64-bit key
//                                   key = (~ordered(score)) << 32 | (anchor * nc + class)
//                               so ascending key order == descending score with ties broken by the
//                               reference's row order (== stable descending sort), and every key is unique:
//                               the result is independent of the (atomic) compaction order.
// Kernel 2  nms_select_kernel   one CTA per image: shared-memory bitonic sort of the keys (radix-select
//                               rounds first when there are more than SORT_CAP candidates, which also
//                               implements the max_nms top-k), then greedy suppression in sorted order, 32
//                               candidates (one per lane) at a time: all 32 warps test them against their share
//                               of the kept list, warp 0 resolves the block's 32 x 32 suppression matrix with
//                               register shuffles and appends the survivors; stops at max_det survivors.
//                               Images whose classes are provably separated by the class offsets take the
//                               class-wise path instead (select_classwise).
// Priors (ops.py labels=, the validator's save_hybrid): label row l of image b is the virtual anchor A + l with
// score 1.0 at its class, its box read from the packed label buffer (MODE 2 of the select kernel).  Its keys
// sort after every anchor key of equal score, which is the reference's row order (labels appended after the
// anchors), so every stage downstream treats the priors exactly like anchors.
// IoU arithmetic follows torchvision's CPU kernel operation by operation (no FMA contraction, same
// std::max/std::min operand order, fp32 IoU compared against the double threshold).
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include "common.cuh"

namespace yl {

constexpr int kSelThreads = 1024;
constexpr int kSortCap = 16384;  // keys sorted in shared memory per round
constexpr int kChunk = 512;      // candidates resolved per bitmask round
constexpr int kMaskWords = kChunk / 32;


// ---------------------------------------------------------------------------------------------- filter
template <int VEC, bool MULTI>
__global__ void __launch_bounds__(256) nms_filter_kernel(const float* __restrict__ pred, int nc, int A, float conf,
                                                         const int32_t* __restrict__ classes, int n_classes,
                                                         unsigned long long cap,
                                                         uint32_t* __restrict__ counts,
                                                         unsigned long long* __restrict__ keys) {
    __shared__ uint32_t cmask[32];  // class filter bitmask (nc <= 1024)
    const int b = blockIdx.y;
    if (n_classes > 0) {
        if (threadIdx.x < 32) cmask[threadIdx.x] = 0;
        __syncthreads();
        for (int i = threadIdx.x; i < n_classes; i += blockDim.x) {
            const int c = classes[i];
            if (c >= 0 && c < nc) atomicOr(&cmask[c >> 5], 1u << (c & 31));
        }
        __syncthreads();
    }
    const int lane = threadIdx.x & 31;
    const int a0 = (blockIdx.x * blockDim.x + threadIdx.x) * VEC;
    const bool in_range = a0 < A;
    const float* base = pred + ((long long)b * (4 + nc) + 4) * A + a0;
    unsigned long long* kout = keys + (unsigned long long)b * cap;

    float best[VEC];
    int bestc[VEC];
#pragma unroll
    for (int v = 0; v < VEC; ++v) {
        best[v] = -INFINITY;
        bestc[v] = 0;
    }

#pragma unroll 8
    for (int c = 0; c < nc; ++c) {
        float s[VEC];
        if (in_range) {
            if (VEC == 4) {
                const float4 t = __ldg(reinterpret_cast<const float4*>(base + (long long)c * A));
                s[0] = t.x; s[1 % VEC] = t.y; s[2 % VEC] = t.z; s[3 % VEC] = t.w;
            } else {
                s[0] = __ldg(base + (long long)c * A);
            }
        } else {
#pragma unroll
            for (int v = 0; v < VEC; ++v) s[v] = -INFINITY;
        }
        if (!MULTI) {
#pragma unroll
            for (int v = 0; v < VEC; ++v)
                if (s[v] > best[v]) {  // strict: ties keep the lowest class index (torch.max)
                    best[v] = s[v];
                    bestc[v] = c;
                }
        } else {
            const bool cls_ok = n_classes == 0 || ((cmask[c >> 5] >> (c & 31)) & 1u);
#pragma unroll
            for (int v = 0; v < VEC; ++v) {
                const bool emit = in_range && cls_ok && (s[v] > conf);
                const unsigned m = __ballot_sync(0xffffffffu, emit);
                if (m) {
                    uint32_t pos0 = 0;
                    if (lane == 0) pos0 = atomicAdd(&counts[b], (uint32_t)__popc(m));
                    pos0 = __shfl_sync(0xffffffffu, pos0, 0);
                    if (emit) {
                        const uint32_t idx = (uint32_t)(a0 + v) * (uint32_t)nc + (uint32_t)c;
                        kout[pos0 + __popc(m & ((1u << lane) - 1u))] =
                            ((unsigned long long)score_to_desc(s[v]) << 32) | idx;
                    }
                }
            }
        }
    }
    if (!MULTI) {
#pragma unroll
        for (int v = 0; v < VEC; ++v) {
            bool emit = in_range && (best[v] > conf);
            if (emit && n_classes > 0) emit = (cmask[bestc[v] >> 5] >> (bestc[v] & 31)) & 1u;
            const unsigned m = __ballot_sync(0xffffffffu, emit);
            if (m) {
                uint32_t pos0 = 0;
                if (lane == 0) pos0 = atomicAdd(&counts[b], (uint32_t)__popc(m));
                pos0 = __shfl_sync(0xffffffffu, pos0, 0);
                if (emit) {
                    const uint32_t idx = (uint32_t)(a0 + v) * (uint32_t)nc + (uint32_t)bestc[v];
                    kout[pos0 + __popc(m & ((1u << lane) - 1u))] =
                        ((unsigned long long)score_to_desc(best[v]) << 32) | idx;
                }
            }
        }
    }
}

// Candidates of the priors of image b (blockIdx.x), appended after the filter kernel's: a prior is a one-hot row (1.0
// at its class), so both label modes give exactly one candidate (1.0, cls), kept when 1.0 > conf (checked by the
// caller) and the class filter admits it.  Class ids are range-checked on the host.
__global__ void nms_prior_keys_kernel(const int32_t* __restrict__ lab_cls, const int32_t* __restrict__ lab_off, int nc,
                                      int A, const int32_t* __restrict__ classes, int n_classes, unsigned long long cap,
                                      uint32_t* __restrict__ counts, unsigned long long* __restrict__ keys) {
    const int b = blockIdx.x;
    const int l0 = lab_off[b], nl = lab_off[b + 1] - l0;
    for (int l = threadIdx.x; l < nl; l += blockDim.x) {
        const int c = lab_cls[l0 + l];
        bool keep = n_classes == 0;
        for (int i = 0; i < n_classes && !keep; ++i) keep = classes[i] == c;
        if (!keep) continue;
        const uint32_t idx = (uint32_t)(A + l) * (uint32_t)nc + (uint32_t)c;
        keys[(unsigned long long)b * cap + atomicAdd(&counts[b], 1u)] = ((unsigned long long)score_to_desc(1.f) << 32) | idx;
    }
}

// keys for yl_nms_boxes: every box is a candidate
__global__ void nms_boxes_keys_kernel(const float* __restrict__ scores, int n, unsigned long long* __restrict__ keys,
                                      uint32_t* __restrict__ counts) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) keys[i] = ((unsigned long long)score_to_desc(scores[i]) << 32) | (uint32_t)i;
    if (i == 0) counts[0] = (uint32_t)n;
}

// ---------------------------------------------------------------------------------------------- select
struct SelParams {
    const float* pred;   // MODE 0 / 2: (B, 4+nc, A) xywh+scores.  MODE 1: boxes (n,4) xyxy
    int nc, A;
    unsigned long long cap;
    const uint32_t* counts;
    const unsigned long long* keys;
    float thr;           // largest float <= double iou threshold
    double thr_mid;      // midpoint of thr and the next float above it (exact in double)
    int thr_tie_up;      // a quotient exactly at thr_mid rounds (ties-to-even) to the float ABOVE thr
    float max_wh;        // class offset scale (0 when agnostic)
    int max_det, max_nms;
    int kept_in_smem;
    int classwise;       // allow the per-class path (A/B switch YL_NMS_CLASSWISE, default on)
    long long* dbg;      // optional [B][8] phase cycle counters (tools/nms_phases.py); NULL in production
    float* kept_ws;      // global kept-list storage when max_det is large: [B][max_det][5] + keys
    unsigned long long* kept_keys_ws;
    float* out;          // MODE 0: (B, max_det, 6)
    int32_t* out_counts;
    long long* keep;     // MODE 1: int64[n]
    const float* lab_xywh;    // MODE 2: priors (L, 4) (cx, cy, w, h); image b owns rows [lab_off[b], lab_off[b+1])
    const int32_t* lab_off;
};

// torchvision CPU: suppressed iff inter / (area_i + area_j - inter) > thr, i = kept (earlier) box; every
// operation is an individually rounded fp32 op (no FMA contraction), the quotient is correctly rounded.
// The division itself is avoided: with t+ the float after thr and mid = (thr + t+) / 2,
//     RN(inter / uni) > thr  <=>  RN(inter / uni) >= t+  <=>  inter / uni > mid  (or == mid when the tie rounds up)
// and for uni > 0 that is inter > mid * uni, which is exact in double (25-bit x 24-bit significands).
struct IouThr {
    float thr;
    double mid;
    int tie_up;
};
__device__ __forceinline__ bool iou_suppresses(const float4 bi, float ai, const float4 bj, float aj, const IouThr t) {
    const float xx1 = (bi.x < bj.x) ? bj.x : bi.x;  // std::max(ix1, x1[j])
    const float yy1 = (bi.y < bj.y) ? bj.y : bi.y;
    const float xx2 = (bj.z < bi.z) ? bj.z : bi.z;  // std::min(ix2, x2[j])
    const float yy2 = (bj.w < bi.w) ? bj.w : bi.w;
    const float dw = __fsub_rn(xx2, xx1), dh = __fsub_rn(yy2, yy1);
    const float w = (0.f < dw) ? dw : 0.f;  // std::max(0, xx2 - xx1)
    const float h = (0.f < dh) ? dh : 0.f;
    const float inter = __fmul_rn(w, h);
    // disjoint boxes (the common case once classes are offset apart): inter == +0, so ovr is 0 or NaN (0/0) and
    // `ovr > thr` is false for every thr >= 0.  A NaN inter fails this test and takes the division below.
    if (inter == 0.f) return false;
    const float uni = __fsub_rn(__fadd_rn(ai, aj), inter);
    if (!(inter > 0.f) || !(uni > 0.f) || isinf(inter) || isinf(uni))
        return __fdiv_rn(inter, uni) > t.thr;  // NaN / inf / non-positive union: the reference's own arithmetic
    const double lhs = (double)inter, rhs = t.mid * (double)uni;
    return t.tie_up ? (lhs >= rhs) : (lhs > rhs);
}

// (cx, cy, w, h) of virtual anchor a >= A of image b (MODE 2): prior row a - A of the image
__device__ __forceinline__ float4 load_prior(const SelParams& p, int b, int a) {
    const float* q = p.lab_xywh + ((long long)__ldg(p.lab_off + b) + (a - p.A)) * 4;
    return make_float4(__ldg(q), __ldg(q + 1), __ldg(q + 2), __ldg(q + 3));
}

// The global loads of fetch_box alone (so a caller can put other work between the loads and their use) ...
template <int MODE>
__device__ __forceinline__ float4 fetch_raw(const SelParams& p, int b, unsigned long long key) {
    const uint32_t idx = (uint32_t)(key & 0xffffffffull);
    if (MODE != 1) {
        const int a = (int)(idx / (uint32_t)p.nc);
        if (MODE == 2 && a >= p.A) return load_prior(p, b, a);
        const float* q = p.pred + (long long)b * (4 + p.nc) * p.A + a;
        return make_float4(__ldg(q), __ldg(q + p.A), __ldg(q + 2 * (long long)p.A), __ldg(q + 3 * (long long)p.A));
    }
    return __ldg(reinterpret_cast<const float4*>(p.pred) + idx);
}
// ... and the arithmetic: offset box (the one NMS works on) + its area, from the raw values (cx, cy, w, h | xyxy)
template <int MODE>
__device__ __forceinline__ void finish_box(const SelParams& p, unsigned long long key, const float4 v, float4* off, float* area) {
    if (MODE != 1) {
        const uint32_t idx = (uint32_t)(key & 0xffffffffull);
        const int a = (int)(idx / (uint32_t)p.nc);
        const int c = (int)(idx - (uint32_t)a * (uint32_t)p.nc);
        const float hw = v.z * 0.5f, hh = v.w * 0.5f;
        const float o = __fmul_rn((float)c, p.max_wh);
        off->x = __fadd_rn(__fsub_rn(v.x, hw), o);
        off->y = __fadd_rn(__fsub_rn(v.y, hh), o);
        off->z = __fadd_rn(__fadd_rn(v.x, hw), o);
        off->w = __fadd_rn(__fadd_rn(v.y, hh), o);
    } else {
        *off = v;
    }
    *area = __fmul_rn(__fsub_rn(off->z, off->x), __fsub_rn(off->w, off->y));
}

template <int MODE>
__device__ __forceinline__ void fetch_box(const SelParams& p, int b, unsigned long long key, float4* raw, float4* off,
                                          float* area, float* score, int* cls) {
    const uint32_t idx = (uint32_t)(key & 0xffffffffull);
    *score = desc_to_score((uint32_t)(key >> 32));
    if (MODE != 1) {
        const int a = (int)(idx / (uint32_t)p.nc);
        const int c = (int)(idx - (uint32_t)a * (uint32_t)p.nc);
        float cx, cy, w, h;
        if (MODE == 2 && a >= p.A) {
            const float4 v = load_prior(p, b, a);
            cx = v.x, cy = v.y, w = v.z, h = v.w;
        } else {
            const float* q = p.pred + (long long)b * (4 + p.nc) * p.A + a;
            cx = __ldg(q), cy = __ldg(q + p.A), w = __ldg(q + 2 * (long long)p.A), h = __ldg(q + 3 * (long long)p.A);
        }
        const float hw = w * 0.5f, hh = h * 0.5f;  // x[..., 2:] / 2 (exact)
        raw->x = __fsub_rn(cx, hw);
        raw->y = __fsub_rn(cy, hh);
        raw->z = __fadd_rn(cx, hw);
        raw->w = __fadd_rn(cy, hh);
        const float o = __fmul_rn((float)c, p.max_wh);  // x[:, 5:6] * max_wh
        off->x = __fadd_rn(raw->x, o);
        off->y = __fadd_rn(raw->y, o);
        off->z = __fadd_rn(raw->z, o);
        off->w = __fadd_rn(raw->w, o);
        *cls = c;
    } else {
        const float4 t = __ldg(reinterpret_cast<const float4*>(p.pred) + idx);
        *raw = t;
        *off = t;
        *cls = 0;
    }
    *area = __fmul_rn(__fsub_rn(off->z, off->x), __fsub_rn(off->w, off->y));
}

// ascending keys == descending score: in-place bitonic sort of skeys[0..P), P a power of two
__device__ __forceinline__ void block_bitonic_sort(unsigned long long* skeys, int P, int tid) {
    for (int k = 2; k <= P; k <<= 1)
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int i = tid; i < P; i += kSelThreads) {
                const int ixj = i ^ j;
                if (ixj > i) {
                    const unsigned long long x = skeys[i], y = skeys[ixj];
                    const bool up = (i & k) == 0;
                    if ((x > y) == up) {
                        skeys[i] = y;
                        skeys[ixj] = x;
                    }
                }
            }
            __syncthreads();
        }
}

// Coarse score bin of a key, monotone in the key order (smaller key = higher score = smaller bin).  Used to cut
// a large candidate list into rounds of ~kRoundTarget best candidates without sorting everything: with
// max_det = 300 the greedy scan almost always finishes inside the first round.
constexpr int kBins = 4096;
constexpr int kRoundTarget = 1024;
constexpr int kBinRoundMax = 4096;                // a bin round larger than this switches the image to radix rounds
constexpr int kDirectSort = 2048;                 // at most this many candidates: sort them all directly
__device__ __forceinline__ int key_bin(unsigned long long k) {
    const float t = desc_to_score((uint32_t)(k >> 32)) * (float)kBins;
    const int b = t >= (float)(kBins - 1) ? (kBins - 1) : (t > 0.f ? (int)t : 0);
    return (kBins - 1) - b;
}


// ---------------------------------------------------------------------------------------------- class-wise select
// With class offsets (ops.py:258, 264: boxes + cls * max_wh) two boxes of DIFFERENT classes cannot overlap as long as
// the x extent of all candidates of the image is shorter than max_wh: their offset x intervals are then disjoint, so
// inter == 0 and torchvision's `iou > thr` is false whatever the boxes are.  Greedy NMS over the whole list is then
// exactly one independent greedy NMS per class followed by a merge of the survivors in score order — the O(n^2) pairwise
// work shrinks by the number of classes and the serial dependency chains become one short chain per class, resolved by
// different warps in parallel.  Taken when the image has at most kCwCap candidates, no class more than kCwMaxSeg of
// them, and the extent test holds; everything else (agnostic NMS, max_nms cuts, huge candidate lists) runs the general
// path below.  Both paths produce identical results (the arithmetic per pair is the same function).
constexpr int kCwCap = 4096;
constexpr int kCwMaxSeg = 256;

template <int MODE>
__device__ __forceinline__ bool select_classwise(const SelParams& p, int b, int n, const unsigned long long* gkeys,
                                                 unsigned char* sm, unsigned long long* kept_keys, int* nk_out) {
    // the 128 KB key area of the general path, re-carved: sort keys | offset boxes | areas | keep flags
    unsigned long long* key2 = reinterpret_cast<unsigned long long*>(sm);                    // [kCwCap]    32 KB
    float4* obox = reinterpret_cast<float4*>(key2 + kCwCap);                                 // [kCwCap]    64 KB
    float* oarea = reinterpret_cast<float*>(obox + kCwCap);                                  // [kCwCap]    16 KB
    unsigned char* keepflag = reinterpret_cast<unsigned char*>(oarea + kCwCap);              // [kCwCap]     4 KB
    int* seg_s = reinterpret_cast<int*>(keepflag + kCwCap);                                  // [1024]       4 KB
    int* seg_e = seg_s + 1024;                                                               // [1024]       4 KB
    unsigned long long* kbuf = reinterpret_cast<unsigned long long*>(sm + (size_t)kSortCap * 8);   // [4096] (mask area)
    int* misc = reinterpret_cast<int*>(sm + (size_t)kSortCap * 8 + (size_t)kChunk * kMaskWords * 4 +
                                       (size_t)kChunk * (16 + 4 + 4) + 256 * 4);             // [64]
    float* red = reinterpret_cast<float*>(sm + (size_t)kSortCap * 8 + (size_t)kChunk * kMaskWords * 4);   // [64] (cbox area)
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t nc = (uint32_t)p.nc;

    // ---- 1. keys regrouped as (class | descending score | anchor): one sort gives per-class score order
    int P = 32;
    while (P < n) P <<= 1;
    for (int i = tid; i < P; i += kSelThreads) {
        unsigned long long k2 = ~0ull;
        if (i < n) {
            const unsigned long long k = gkeys[i];
            const uint32_t idx = (uint32_t)(k & 0xffffffffull);
            const uint32_t a = idx / nc, c = idx - a * nc;
            k2 = ((unsigned long long)c << 54) | ((k >> 32) << 22) | (unsigned long long)a;
        }
        key2[i] = k2;
        if (i < kCwCap) keepflag[i] = 0;
    }
    for (int i = tid; i < 1024; i += kSelThreads) {
        seg_s[i] = 0;
        seg_e[i] = 0;
    }
    if (tid == 0) {
        misc[0] = 0;   // fallback flag
        misc[1] = 0;   // kept counter
    }
    __syncthreads();
    block_bitonic_sort(key2, P, tid);

    // ---- 2. boxes of the sorted candidates, class segments, extent of the raw x coordinates
    float xmin = INFINITY, xmax = -INFINITY;
    bool bad = false;
    for (int i = tid; i < n; i += kSelThreads) {
        const unsigned long long k2 = key2[i];
        const uint32_t c = (uint32_t)(k2 >> 54), a = (uint32_t)(k2 & 0x3fffffull);
        const unsigned long long k = (((k2 >> 22) & 0xffffffffull) << 32) | (unsigned long long)(a * nc + c);
        float4 rb, ob;
        float ar, sc;
        int cl;
        fetch_box<MODE>(p, b, k, &rb, &ob, &ar, &sc, &cl);
        obox[i] = ob;
        oarea[i] = ar;
        if (!(rb.x == rb.x) || !(rb.z == rb.z)) bad = true;   // NaN: the extent argument does not apply
        xmin = fminf(xmin, fminf(rb.x, rb.z));
        xmax = fmaxf(xmax, fmaxf(rb.x, rb.z));
        const uint32_t cprev = i > 0 ? (uint32_t)(key2[i - 1] >> 54) : 0xffffffffu;
        const uint32_t cnext = i + 1 < n ? (uint32_t)(key2[i + 1] >> 54) : 0xffffffffu;
        if (c != cprev) seg_s[c] = i;
        if (c != cnext) {
            seg_e[c] = i + 1;
        }
    }
    for (int o = 16; o > 0; o >>= 1) {
        xmin = fminf(xmin, __shfl_xor_sync(0xffffffffu, xmin, o));
        xmax = fmaxf(xmax, __shfl_xor_sync(0xffffffffu, xmax, o));
    }
    if (lane == 0) {
        red[warp] = xmin;
        red[32 + warp] = xmax;
    }
    if (bad) misc[0] = 1;
    __syncthreads();
    if (tid < 32) {
        float lo = red[tid], hi = red[32 + tid];
        for (int o = 16; o > 0; o >>= 1) {
            lo = fminf(lo, __shfl_xor_sync(0xffffffffu, lo, o));
            hi = fmaxf(hi, __shfl_xor_sync(0xffffffffu, hi, o));
        }
        // offset intervals of different classes are disjoint iff the raw extent is shorter than the class pitch
        if (tid == 0 && !(hi - lo < p.max_wh)) misc[0] = 1;
    }
    for (int c = tid; c < (int)nc; c += kSelThreads)
        if (seg_e[c] - seg_s[c] > kCwMaxSeg) misc[0] = 1;
    __syncthreads();
    if (misc[0]) return false;   // (uniform) the general path redoes the image from the global keys

    // ---- 3. one greedy NMS per class, classes spread over the warps
    const IouThr thr = {p.thr, p.thr_mid, p.thr_tie_up};
    for (int c = warp; c < (int)nc; c += kSelThreads / 32) {
        const int s0 = seg_s[c], len = seg_e[c] - s0;
        int kc = 0;   // kept of this class (a class cannot place more than max_det boxes in the final list)
        for (int q0 = 0; q0 < len && kc < p.max_det; q0 += 32) {
            const int j = q0 + lane;
            const bool valid = j < len;
            const float4 bj = valid ? obox[s0 + j] : make_float4(0.f, 0.f, 0.f, 0.f);
            const float aj = valid ? oarea[s0 + j] : 0.f;
            bool alive = valid;
            // against the boxes of this class kept in earlier blocks (better scores)
            for (int t = 0; t < q0; ++t) {
                if (!keepflag[s0 + t]) continue;                       // uniform: one shared byte
                if (alive && iou_suppresses(obox[s0 + t], oarea[s0 + t], bj, aj, thr)) alive = false;
                if (!__any_sync(0xffffffffu, alive)) break;
            }
            // inside the block: row i = the candidates box i would suppress
            const uint32_t alive_mask = __ballot_sync(0xffffffffu, alive);
            uint32_t rowbits = 0;
            for (int i = 0; i < 32; ++i) {
                if (!((alive_mask >> i) & 1u)) continue;               // uniform
                float4 bi;
                bi.x = __shfl_sync(0xffffffffu, bj.x, i);
                bi.y = __shfl_sync(0xffffffffu, bj.y, i);
                bi.z = __shfl_sync(0xffffffffu, bj.z, i);
                bi.w = __shfl_sync(0xffffffffu, bj.w, i);
                const float ai = __shfl_sync(0xffffffffu, aj, i);
                const bool sup = alive && lane > i && iou_suppresses(bi, ai, bj, aj, thr);
                const uint32_t bits = __ballot_sync(0xffffffffu, sup);
                if (lane == i) rowbits = bits;
            }
            uint32_t live = alive_mask, keep = 0;
            int room = p.max_det - kc;
            while (live && room > 0) {
                const int l = __ffs(live) - 1;
                keep |= 1u << l;
                --room;
                live &= ~(__shfl_sync(0xffffffffu, rowbits, l) | (1u << l));
            }
            if (valid && ((keep >> lane) & 1u)) keepflag[s0 + j] = 1;
            kc += __popc(keep);
            __syncwarp();
        }
    }
    __syncthreads();

    // ---- 4. survivors of all classes back in global score order; the best max_det are the result (ops.py:266)
    for (int i = tid; i < n; i += kSelThreads) {
        if (!keepflag[i]) continue;
        const unsigned long long k2 = key2[i];
        const uint32_t c = (uint32_t)(k2 >> 54), a = (uint32_t)(k2 & 0x3fffffull);
        kbuf[atomicAdd(&misc[1], 1)] = (((k2 >> 22) & 0xffffffffull) << 32) | (unsigned long long)(a * nc + c);
    }
    __syncthreads();
    const int K = misc[1];
    int P2 = 32;
    while (P2 < K) P2 <<= 1;
    for (int i = K + tid; i < P2; i += kSelThreads) kbuf[i] = ~0ull;
    __syncthreads();
    block_bitonic_sort(kbuf, P2, tid);
    const int nk = K < p.max_det ? K : p.max_det;
    for (int r = tid; r < nk; r += kSelThreads) kept_keys[r] = kbuf[r];
    __syncthreads();
    *nk_out = nk;
    return true;
}

template <int MODE>
__global__ void __launch_bounds__(kSelThreads, 1) nms_select_kernel(const SelParams p) {
    extern __shared__ __align__(16) unsigned char sm[];
    unsigned long long* skeys = reinterpret_cast<unsigned long long*>(sm);              // [kSortCap]
    uint32_t* mask = reinterpret_cast<uint32_t*>(skeys + kSortCap);                    // [kChunk][kMaskWords]
    float4* cbox = reinterpret_cast<float4*>(mask + kChunk * kMaskWords);              // [kChunk] compacted
    float* carea = reinterpret_cast<float*>(cbox + kChunk);                            // [kChunk]
    int* csrc = reinterpret_cast<int*>(carea + kChunk);                                // [kChunk]
    uint32_t* hist = reinterpret_cast<uint32_t*>(csrc + kChunk);                       // [256]
    int* misc = reinterpret_cast<int*>(hist + 256);                                    // [64]
    unsigned long long* misc64 = reinterpret_cast<unsigned long long*>(misc + 64);     // [4]
    float* kept_sm = reinterpret_cast<float*>(misc64 + 4);                             // [max_det][5] (optional)

    const int b = blockIdx.x;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const unsigned long long* gkeys = p.keys + (unsigned long long)b * p.cap;
    unsigned long long n64 = p.counts[b];
    if (n64 > p.cap) n64 = p.cap;
    const int n = (int)n64;
    const int n_proc = n < p.max_nms ? n : p.max_nms;

    float* kept = p.kept_in_smem ? kept_sm : (p.kept_ws + (long long)b * p.max_det * 5);
    unsigned long long* kept_keys =
        p.kept_in_smem ? reinterpret_cast<unsigned long long*>(kept_sm + (size_t)p.max_det * 5 + (p.max_det & 1))
                       : (p.kept_keys_ws + (long long)b * p.max_det);

    int nk = 0;          // kept so far (uniform across the block)
    int processed = 0;   // candidates consumed in sorted order
    // per-class greedy NMS when the class offsets provably separate the classes (see select_classwise)
    bool classwise_done = false;
    // (anchors + priors of the image must fit the 22-bit anchor field of the regrouped keys)
    const int n_anchors = p.A + (MODE == 2 ? p.lab_off[b + 1] - p.lab_off[b] : 0);
    if (MODE != 1 && p.classwise && p.max_wh > 0.f && n >= 1 && n <= kCwCap && n <= p.max_nms && p.nc <= 1024 &&
        n_anchors < (1 << 22) && p.kept_in_smem)
        classwise_done = select_classwise<MODE>(p, b, n, gkeys, sm, kept_keys, &nk);
    __syncthreads();
    unsigned long long lo = 0;  // keys <= lo are already consumed (radix rounds)
    const bool single_round = n <= kDirectSort;
    // bin mode: cumulative histogram of the coarse score bins (lives in the tail of the key buffer)
    uint32_t* cum = reinterpret_cast<uint32_t*>(skeys + (kSortCap - kBins / 2));
    bool use_bins = false;
    int bpos = 0;  // bins < bpos are consumed
    if (!single_round) {
        for (int i = tid; i < kBins; i += kSelThreads) cum[i] = 0;
        __syncthreads();
        for (int i = tid; i < n; i += kSelThreads) atomicAdd(&cum[key_bin(gkeys[i])], 1u);
        __syncthreads();
        // block-wide inclusive scan, kBins / kSelThreads (= 4) bins per thread
        constexpr int PER = kBins / kSelThreads;
        uint32_t v[PER], tsum = 0;
#pragma unroll
        for (int i = 0; i < PER; ++i) {
            v[i] = cum[tid * PER + i];
            tsum += v[i];
        }
        uint32_t incl = tsum;
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += t;
        }
        if (lane == 31) hist[warp] = incl;
        use_bins = true;
        __syncthreads();
        if (warp == 0) {
            const uint32_t w = hist[lane];
            uint32_t wi = w;
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t t = __shfl_up_sync(0xffffffffu, wi, o);
                if (lane >= o) wi += t;
            }
            hist[lane] = wi - w;
        }
        __syncthreads();
        uint32_t run = hist[warp] + incl - tsum;
#pragma unroll
        for (int i = 0; i < PER; ++i) {
            run += v[i];
            cum[tid * PER + i] = run;
        }
        __syncthreads();
    }

    if (tid == 0) misc[5] = 0;   // lanes of the current 32-candidate block suppressed by the kept list
    __syncthreads();
    long long tph = clock64(), acc_ph[8] = {0, 0, 0, 0, 0, 0, 0, 0};
#define YL_PH(k)                                   \
    do {                                           \
        if (p.dbg && tid == 0) {                   \
            const long long t_ = clock64();        \
            acc_ph[k] += t_ - tph;                 \
            tph = t_;                              \
        }                                          \
    } while (0)
    YL_PH(0);
    while (!classwise_done && processed < n_proc && nk < p.max_det) {
        int m = n_proc - processed;
        if (m > kSortCap) m = kSortCap;
        int consumed = m;  // candidates this round removes from the unprocessed set
        // ---------------- stage the next m keys (ascending) into shared memory
        if (single_round) {
            for (int i = tid; i < n; i += kSelThreads) skeys[i] = gkeys[i];
            int P = 32;
            while (P < n) P <<= 1;
            for (int i = n + tid; i < P; i += kSelThreads) skeys[i] = ~0ull;
            __syncthreads();
            block_bitonic_sort(skeys, P, tid);
        } else {
            bool staged = false;
            if (use_bins) {
                // the best ~kRoundTarget unconsumed candidates: bins [bpos, e)
                if (tid == 0) {
                    const uint32_t base = bpos ? cum[bpos - 1] : 0u;
                    int lo_b = bpos, hi_b = kBins - 1;  // smallest e-1 with cum[e-1] - base >= target (or last bin)
                    while (lo_b < hi_b) {
                        const int mid = (lo_b + hi_b) >> 1;
                        if (cum[mid] - base >= (uint32_t)kRoundTarget) hi_b = mid; else lo_b = mid + 1;
                    }
                    misc[0] = lo_b + 1;
                    misc[1] = (int)(cum[lo_b] - base);
                    misc[2] = 0;
                }
                __syncthreads();
                const int e = misc[0];
                const int mr = misc[1];
                if (mr <= kBinRoundMax) {
                    for (int i0 = 0; i0 < n; i0 += kSelThreads) {
                        const int i = i0 + tid;
                        unsigned long long k = 0;
                        bool take = false;
                        if (i < n) {
                            k = gkeys[i];
                            const int kb = key_bin(k);
                            take = kb >= bpos && kb < e;
                        }
                        const unsigned bal = __ballot_sync(0xffffffffu, take);
                        if (bal) {
                            int pos0 = 0;
                            if (lane == 0) pos0 = atomicAdd(&misc[2], __popc(bal));
                            pos0 = __shfl_sync(0xffffffffu, pos0, 0);
                            if (take) skeys[pos0 + __popc(bal & ((1u << lane) - 1u))] = k;
                        }
                    }
                    __syncthreads();
                    int P = 32;
                    while (P < mr) P <<= 1;
                    for (int i = mr + tid; i < P; i += kSelThreads) skeys[i] = ~0ull;
                    __syncthreads();
                    block_bitonic_sort(skeys, P, tid);
                    bpos = e;
                    lo = skeys[mr - 1];  // largest key consumed so far (a later radix round resumes above it)
                    consumed = mr;
                    m = mr < (n_proc - processed) ? mr : (n_proc - processed);  // max_nms cut inside the round
                    staged = true;
                } else {
                    // the score bins are too coarse here (many near-equal scores): exact radix rounds from now on;
                    // every key of the bins consumed so far is <= lo, every other key is > lo
                    use_bins = false;
                    __syncthreads();  // misc[] is rewritten below
                }
            }
            if (!staged) {
                // radix select: T = m-th smallest key among keys > lo (8 passes of 8 bits, MSD first); a round takes
                // the next kRoundTarget candidates, so a greedy scan that fills max_det early never sorts the rest
                if (m > kRoundTarget) m = kRoundTarget;
                consumed = m;
                unsigned long long prefix = 0, pmask = 0;
                int remaining = m;
                for (int pass = 0; pass < 8; ++pass) {
                    const int shift = 56 - 8 * pass;
                    if (tid < 256) hist[tid] = 0;
                    __syncthreads();
                    for (int i = tid; i < n; i += kSelThreads) {
                        const unsigned long long k = gkeys[i];
                        if (k > lo && (k & pmask) == prefix) atomicAdd(&hist[(uint32_t)(k >> shift) & 0xffu], 1u);
                    }
                    __syncthreads();
                    if (warp == 0) {
                        // digit d with count(digits < d) < remaining <= count(digits <= d): 8 bins per lane
                        uint32_t c[8], ls = 0;
#pragma unroll
                        for (int i = 0; i < 8; ++i) {
                            c[i] = hist[lane * 8 + i];
                            ls += c[i];
                        }
                        uint32_t incl = ls;
                        for (int o = 1; o < 32; o <<= 1) {
                            const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
                            if (lane >= o) incl += t;
                        }
                        const unsigned hit = __ballot_sync(0xffffffffu, incl >= (uint32_t)remaining);
                        const int src = hit ? (__ffs(hit) - 1) : 31;
                        if (lane == src) {
                            uint32_t acc = incl - ls;
                            int d = 0;
                            for (; d < 7; ++d) {
                                if (acc + c[d] >= (uint32_t)remaining) break;
                                acc += c[d];
                            }
                            misc[0] = lane * 8 + d;
                            misc[1] = remaining - (int)acc;
                        }
                    }
                    __syncthreads();
                    prefix |= (unsigned long long)misc[0] << shift;
                    pmask |= 0xffull << shift;
                    remaining = misc[1];
                    __syncthreads();
                }
                const unsigned long long T = prefix;
                if (tid == 0) misc[2] = 0;
                __syncthreads();
                for (int i = tid; i < n; i += kSelThreads) {
                    const unsigned long long k = gkeys[i];
                    if (k > lo && k <= T) skeys[atomicAdd(&misc[2], 1)] = k;
                }
                __syncthreads();
                // exactly m keys were gathered (keys are unique); sort them
                int P = 32;
                while (P < m) P <<= 1;
                for (int i = m + tid; i < P; i += kSelThreads) skeys[i] = ~0ull;
                __syncthreads();
                block_bitonic_sort(skeys, P, tid);
                lo = T;
            }
        }

        YL_PH(1);   // round staging: gather + sort
        // ---------------- greedy suppression over skeys[0..m), 32 candidates (one per lane) at a time, in score order
        // Before the block barrier every warp (i) tests the block's candidates against ITS share of the kept list (kept
        // boxes warp, warp + 32, ...) and ORs the suppressed lanes into one shared word, (ii) computes row `warp` of the
        // block's 32 x 32 suppression matrix (candidate `warp` against the later candidates, one IoU per lane) and
        // (iii) issues the global loads of the NEXT block's boxes.  After it warp 0 runs the greedy pass over the matrix
        // rows of the surviving candidates and appends the kept ones.  No speculative pairwise work beyond 32 x 32,
        // two block barriers per 32 candidates, the scan stops at max_det kept boxes.
        const IouThr thr = {p.thr, p.thr_mid, p.thr_tie_up};
        bool valid = lane < m;
        float4 ob = make_float4(0.f, 0.f, 0.f, 0.f), rb;
        float ar = 0.f, sc;
        int cl;
        unsigned long long key = 0;
        if (valid) {
            key = skeys[lane];
            fetch_box<MODE>(p, b, key, &rb, &ob, &ar, &sc, &cl);
        }
        for (int s0 = 0; s0 < m && nk < p.max_det; s0 += 32) {
            // (iii) next block's candidates: only the loads are issued here, they fly under (i) and (ii)
            const bool nvalid = s0 + 32 + lane < m;
            float4 nraw = make_float4(0.f, 0.f, 0.f, 0.f);
            unsigned long long nkey = 0;
            if (nvalid) {
                nkey = skeys[s0 + 32 + lane];
                nraw = fetch_raw<MODE>(p, b, nkey);
            }
            // (i)
            bool dead = false;
            for (int i = warp; i < nk; i += kSelThreads / 32) {
                const float4 kb = make_float4(kept[i * 5 + 0], kept[i * 5 + 1], kept[i * 5 + 2], kept[i * 5 + 3]);
                if (valid && !dead && iou_suppresses(kb, kept[i * 5 + 4], ob, ar, thr)) dead = true;
            }
            const unsigned dbits = __ballot_sync(0xffffffffu, dead);
            if (lane == 0 && dbits) atomicOr(reinterpret_cast<unsigned*>(&misc[5]), dbits);
            // (ii) row `warp`
            {
                float4 bi;
                bi.x = __shfl_sync(0xffffffffu, ob.x, warp);
                bi.y = __shfl_sync(0xffffffffu, ob.y, warp);
                bi.z = __shfl_sync(0xffffffffu, ob.z, warp);
                bi.w = __shfl_sync(0xffffffffu, ob.w, warp);
                const float ai = __shfl_sync(0xffffffffu, ar, warp);
                const bool sup = valid && lane > warp && (s0 + warp < m) && iou_suppresses(bi, ai, ob, ar, thr);
                const unsigned bits = __ballot_sync(0xffffffffu, sup);
                if (lane == 0) misc[8 + warp] = (int)bits;
            }
            __syncthreads();
            YL_PH(2);   // vs kept + block matrix row
            if (warp == 0) {
                const uint32_t alive_mask = __ballot_sync(0xffffffffu, valid) & ~(uint32_t)misc[5];
                const uint32_t rowbits = (uint32_t)misc[8 + lane];
                uint32_t live = alive_mask, keep = 0;
                int room = p.max_det - nk;
                while (live && room > 0) {
                    const int l = __ffs(live) - 1;
                    keep |= 1u << l;
                    --room;
                    live &= ~(__shfl_sync(0xffffffffu, rowbits, l) | (1u << l));
                }
                if ((keep >> lane) & 1u) {
                    const int pos = nk + __popc(keep & ((1u << lane) - 1u));
                    kept[pos * 5 + 0] = ob.x;
                    kept[pos * 5 + 1] = ob.y;
                    kept[pos * 5 + 2] = ob.z;
                    kept[pos * 5 + 3] = ob.w;
                    kept[pos * 5 + 4] = ar;
                    kept_keys[pos] = key;
                }
                if (lane == 0) {
                    misc[4] = nk + __popc(keep);
                    misc[5] = 0;
                }
                YL_PH(5);   // greedy pass + append
            }
            __threadfence_block();
            __syncthreads();
            nk = misc[4];
            valid = nvalid;
            key = nkey;
            ob = make_float4(0.f, 0.f, 0.f, 0.f);
            ar = 0.f;
            if (valid) finish_box<MODE>(p, key, nraw, &ob, &ar);
        }
        processed += consumed;
    }
    if (p.dbg && tid == 0) {
        acc_ph[6] = nk;
        acc_ph[7] = processed;
        for (int k = 0; k < 8; ++k) p.dbg[(long long)b * 8 + k] = acc_ph[k];
    }

    // ---------------- emit
    if (MODE != 1) {
        float* o = p.out + (long long)b * p.max_det * 6;
        for (int r = tid; r < p.max_det; r += kSelThreads) {
            float4 rb = make_float4(0, 0, 0, 0), ob;
            float ar, sc = 0.f;
            int cl = 0;
            if (r < nk) fetch_box<MODE>(p, b, kept_keys[r], &rb, &ob, &ar, &sc, &cl);
            o[r * 6 + 0] = rb.x;
            o[r * 6 + 1] = rb.y;
            o[r * 6 + 2] = rb.z;
            o[r * 6 + 3] = rb.w;
            o[r * 6 + 4] = sc;
            o[r * 6 + 5] = (float)cl;
        }
        if (tid == 0) p.out_counts[b] = nk;
    } else {
        for (int r = tid; r < nk; r += kSelThreads) p.keep[r] = (long long)(kept_keys[r] & 0xffffffffull);
        if (tid == 0) p.out_counts[0] = nk;
    }
}

static size_t sel_smem_bytes(int max_det, bool kept_in_smem) {
    size_t s = (size_t)kSortCap * 8 + (size_t)kChunk * kMaskWords * 4 + (size_t)kChunk * (16 + 4 + 4) + 256 * 4 +
               64 * 4 + 4 * 8;
    if (kept_in_smem) s += ((size_t)max_det * 5 + (max_det & 1)) * 4 + (size_t)max_det * 8 + 16;
    return s;
}

static int g_sel_max_smem = 0;
static int g_nms_classwise = 1;   // YL_NMS_CLASSWISE, read once in yl_init
static thread_local long long* g_nms_dbg = nullptr;   // yl_debug_nms_phases

int init_nms() {
    {
        const char* e = getenv("YL_NMS_CLASSWISE");
        g_nms_classwise = (e && *e) ? (atoi(e) != 0) : 1;
    }
    int dev = 0;
    YL_CUDA(cudaGetDevice(&dev));
    YL_CUDA(cudaDeviceGetAttribute(&g_sel_max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
    YL_CUDA(cudaFuncSetAttribute(nms_select_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, g_sel_max_smem));
    YL_CUDA(cudaFuncSetAttribute(nms_select_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, g_sel_max_smem));
    YL_CUDA(cudaFuncSetAttribute(nms_select_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, g_sel_max_smem));
    return YL_OK;
}

static float thr_to_float(double thr) {
    // largest float f with (double)f <= thr: then  (double)ovr > thr  <=>  ovr > f  for every float ovr
    float f = (float)thr;
    if ((double)f > thr) f = nextafterf(f, -INFINITY);
    return f;
}

// Rounding boundary between thr and the next float above it, and which way an exact tie goes (round-to-nearest-
// even picks the neighbour with an even significand: the upper one iff thr's is odd).
static void thr_midpoint(float thr, double* mid, int* tie_up) {
    const float up = nextafterf(thr, INFINITY);
    *mid = ((double)thr + (double)up) * 0.5;  // exact: both are floats one ulp apart
    uint32_t bits;
    memcpy(&bits, &thr, 4);
    *tie_up = (int)(bits & 1u);
}

static size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

__global__ void xywh2xyxy_kernel(float* __restrict__ pred, int C, int A, long long total) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const int a = (int)(i % A);
    const long long b = i / A;
    float* q = pred + b * C * A + a;
    const float cx = q[0], cy = q[A], hw = q[2 * (long long)A] * 0.5f, hh = q[3 * (long long)A] * 0.5f;
    q[0] = __fsub_rn(cx, hw);
    q[A] = __fsub_rn(cy, hh);
    q[2 * (long long)A] = __fadd_rn(cx, hw);
    q[3 * (long long)A] = __fadd_rn(cy, hh);
}

__global__ void scale_boxes_kernel(float* __restrict__ dets, const int32_t* __restrict__ counts, int max_det,
                                   const float* __restrict__ params) {
    const int b = blockIdx.x;
    const float gain = params[b * 5 + 0], padx = params[b * 5 + 1], pady = params[b * 5 + 2], w0 = params[b * 5 + 3],
                h0 = params[b * 5 + 4];
    const int n = counts[b];
    for (int r = threadIdx.x; r < n; r += blockDim.x) {
        float* d = dets + ((long long)b * max_det + r) * 6;
        // ops.scale_boxes: subtract pad, divide by gain (true division), clip_boxes clamp
        float x1 = __fdiv_rn(__fsub_rn(d[0], padx), gain), y1 = __fdiv_rn(__fsub_rn(d[1], pady), gain);
        float x2 = __fdiv_rn(__fsub_rn(d[2], padx), gain), y2 = __fdiv_rn(__fsub_rn(d[3], pady), gain);
        d[0] = fminf(fmaxf(x1, 0.f), w0);
        d[1] = fminf(fmaxf(y1, 0.f), h0);
        d[2] = fminf(fmaxf(x2, 0.f), w0);
        d[3] = fminf(fmaxf(y2, 0.f), h0);
    }
}

static int launch_select(const float* pred, int B, int nc, int A, size_t cap, const uint32_t* cand_counts,
                         const unsigned long long* keys, double iou_thres, int agnostic, int max_det, int max_nms,
                         float max_wh, const float* lab_xywh, const int32_t* lab_off, float* out, int32_t* counts,
                         cudaStream_t s) {
    SelParams p;
    p.pred = pred;
    p.nc = nc;
    p.A = A;
    p.lab_xywh = lab_xywh;
    p.lab_off = lab_off;
    p.cap = cap;
    p.counts = cand_counts;
    p.keys = keys;
    p.thr = thr_to_float(iou_thres);
    thr_midpoint(p.thr, &p.thr_mid, &p.thr_tie_up);
    p.max_wh = agnostic ? 0.f : max_wh;
    p.max_det = max_det;
    p.max_nms = max_nms;
    p.kept_in_smem = 1;
    p.classwise = g_nms_classwise;
    p.dbg = yl::g_nms_dbg;
    p.kept_ws = nullptr;
    p.kept_keys_ws = nullptr;
    p.out = out;
    p.out_counts = counts;
    p.keep = nullptr;
    const size_t smem = sel_smem_bytes(max_det, true);
    YL_CHECK((int)smem <= g_sel_max_smem, YL_ERR_UNSUPPORTED, "NMS needs %zu B shared memory (yl_init called?)", smem);
    if (lab_off) nms_select_kernel<2><<<B, kSelThreads, smem, s>>>(p);
    else nms_select_kernel<0><<<B, kSelThreads, smem, s>>>(p);
    YL_LAUNCH_OK("nms_select_kernel");
    return YL_OK;
}

}  // namespace yl

extern "C" {

size_t yl_nms_priors_workspace_bytes(int B, int A, int nc, int multi_label, int max_labels_per_image) {
    if (B <= 0 || A <= 0 || nc <= 0 || max_labels_per_image < 0) return 0;
    // every prior adds at most one candidate (its own class) in either label mode
    const size_t cap = (multi_label ? (size_t)A * nc : (size_t)A) + (size_t)max_labels_per_image;
    size_t s = yl::align_up((size_t)B * 4, 256);   // candidate counters
    s += yl::align_up((size_t)B * cap * 8, 256);   // keys
    return s;
}

size_t yl_nms_workspace_bytes(int B, int A, int nc, int multi_label) {
    return yl_nms_priors_workspace_bytes(B, A, nc, multi_label, 0);
}

int yl_nms_batched_priors(const float* pred, int B, int nc, int A, float conf_thres, double iou_thres,
                          const int32_t* classes_dev, int n_classes, int agnostic, int multi_label, int max_det,
                          int max_nms, float max_wh, const float* label_xywh, const int32_t* label_cls,
                          const int32_t* label_offsets, int max_labels_per_image, void* workspace,
                          size_t workspace_bytes, float* out, int32_t* counts, void* stream) {
    YL_CHECK(pred && out && counts && workspace, YL_ERR_ARG, "null pointer");
    YL_CHECK(B > 0 && nc > 0 && nc <= 1024 && A > 0, YL_ERR_ARG, "bad dims B=%d nc=%d A=%d", B, nc, A);
    YL_CHECK(max_labels_per_image >= 0, YL_ERR_ARG, "negative max_labels_per_image");
    const int L = label_offsets ? max_labels_per_image : 0;
    YL_CHECK(L == 0 || (label_xywh && label_cls), YL_ERR_ARG, "label_xywh / label_cls is NULL");
    YL_CHECK((long long)(A + (long long)L) * nc < (1ll << 32), YL_ERR_ARG, "(A + max_labels_per_image)*nc must fit 32 bits");
    YL_CHECK(max_det > 0 && max_det <= 1024, YL_ERR_ARG, "max_det must be in [1,1024]");
    YL_CHECK(max_nms > 0, YL_ERR_ARG, "max_nms must be positive");
    YL_CHECK(conf_thres >= 0.f && conf_thres <= 1.f && iou_thres >= 0. && iou_thres <= 1., YL_ERR_ARG,
             "thresholds must be in [0,1]");
    YL_CHECK(n_classes == 0 || classes_dev, YL_ERR_ARG, "classes_dev is NULL");
    const size_t need = yl_nms_priors_workspace_bytes(B, A, nc, multi_label, L);
    YL_CHECK(workspace_bytes >= need, YL_ERR_WORKSPACE, "NMS workspace too small: %zu < %zu", workspace_bytes, need);
    cudaStream_t s = (cudaStream_t)stream;
    multi_label = multi_label && nc > 1;
    const int32_t* lab_off = L > 0 ? label_offsets : nullptr;   // no priors: the plain path, launch for launch

    const size_t cap = (multi_label ? (size_t)A * nc : (size_t)A) + (size_t)L;
    uint32_t* cand_counts = reinterpret_cast<uint32_t*>(workspace);
    unsigned long long* keys =
        reinterpret_cast<unsigned long long*>(reinterpret_cast<char*>(workspace) + yl::align_up((size_t)B * 4, 256));
    YL_CUDA(cudaMemsetAsync(cand_counts, 0, (size_t)B * 4, s));

    const bool vec4 = (A % 4 == 0) && ((reinterpret_cast<uintptr_t>(pred) & 15) == 0);
    {
        dim3 grid((unsigned)yl::ceil_div(A, vec4 ? 256 * 4 : 256), (unsigned)B, 1);
#define YL_FILTER(V, M)                                                                                      \
    yl::nms_filter_kernel<V, M><<<grid, 256, 0, s>>>(pred, nc, A, conf_thres, classes_dev, n_classes,          \
                                                     (unsigned long long)cap, cand_counts, keys)
        if (vec4 && multi_label) YL_FILTER(4, true);
        else if (vec4) YL_FILTER(4, false);
        else if (multi_label) YL_FILTER(1, true);
        else YL_FILTER(1, false);
#undef YL_FILTER
    }
    YL_LAUNCH_OK("nms_filter_kernel");
    if (lab_off && 1.f > conf_thres) {
        yl::nms_prior_keys_kernel<<<B, 128, 0, s>>>(label_cls, lab_off, nc, A, classes_dev, n_classes,
                                                    (unsigned long long)cap, cand_counts, keys);
        YL_LAUNCH_OK("nms_prior_keys_kernel");
    }

    return yl::launch_select(pred, B, nc, A, cap, cand_counts, keys, iou_thres, agnostic, max_det, max_nms, max_wh,
                             label_xywh, lab_off, out, counts, s);
}

int yl_nms_batched(const float* pred, int B, int nc, int A, float conf_thres, double iou_thres,
                   const int32_t* classes_dev, int n_classes, int agnostic, int multi_label, int max_det, int max_nms,
                   float max_wh, void* workspace, size_t workspace_bytes, float* out, int32_t* counts, void* stream) {
    return yl_nms_batched_priors(pred, B, nc, A, conf_thres, iou_thres, classes_dev, n_classes, agnostic, multi_label,
                                 max_det, max_nms, max_wh, nullptr, nullptr, nullptr, 0, workspace, workspace_bytes, out,
                                 counts, stream);
}

int yl_debug_nms_phases(long long* device_buf) {
    yl::g_nms_dbg = device_buf;
    return YL_OK;
}

int yl_nms_begin(void* workspace, size_t workspace_bytes, int B, void* stream) {
    YL_CHECK(workspace && B > 0 && workspace_bytes >= (size_t)B * 4, YL_ERR_ARG, "bad nms_begin arguments");
    YL_CUDA(cudaMemsetAsync(workspace, 0, (size_t)B * 4, (cudaStream_t)stream));
    return YL_OK;
}

int yl_nms_select(const float* pred, int B, int nc, int A, double iou_thres, int agnostic, int max_det, int max_nms,
                  float max_wh, void* workspace, size_t workspace_bytes, float* out, int32_t* counts, void* stream) {
    YL_CHECK(pred && out && counts && workspace, YL_ERR_ARG, "null pointer");
    YL_CHECK(B > 0 && nc > 0 && nc <= 1024 && A > 0, YL_ERR_ARG, "bad dims B=%d nc=%d A=%d", B, nc, A);
    YL_CHECK((long long)A * nc < (1ll << 32), YL_ERR_ARG, "A*nc must fit 32 bits");
    YL_CHECK(max_det > 0 && max_det <= 1024, YL_ERR_ARG, "max_det must be in [1,1024]");
    YL_CHECK(max_nms > 0 && iou_thres >= 0. && iou_thres <= 1., YL_ERR_ARG, "bad thresholds");
    YL_CHECK(workspace_bytes >= yl_nms_workspace_bytes(B, A, nc, 0), YL_ERR_WORKSPACE, "NMS workspace too small");
    uint32_t* cand_counts = reinterpret_cast<uint32_t*>(workspace);
    unsigned long long* keys =
        reinterpret_cast<unsigned long long*>(reinterpret_cast<char*>(workspace) + yl::align_up((size_t)B * 4, 256));
    return yl::launch_select(pred, B, nc, A, (size_t)A, cand_counts, keys, iou_thres, agnostic, max_det, max_nms, max_wh,
                             nullptr, nullptr, out, counts, (cudaStream_t)stream);
}

size_t yl_nms_boxes_workspace_bytes(int n) {
    if (n <= 0) return 256;
    return 256 + yl::align_up((size_t)n * 8, 256) + yl::align_up((size_t)n * 5 * 4, 256) +
           yl::align_up((size_t)n * 8, 256);
}

int yl_nms_boxes(const float* boxes, const float* scores, int n, double iou_thres, void* workspace,
                 size_t workspace_bytes, int64_t* keep, int32_t* count, void* stream) {
    YL_CHECK(count && workspace, YL_ERR_ARG, "null pointer");
    YL_CHECK(n >= 0, YL_ERR_ARG, "negative n");
    cudaStream_t s = (cudaStream_t)stream;
    if (n == 0) {
        YL_CUDA(cudaMemsetAsync(count, 0, 4, s));
        return YL_OK;
    }
    YL_CHECK(boxes && scores && keep, YL_ERR_ARG, "null pointer");
    YL_CHECK((reinterpret_cast<uintptr_t>(boxes) & 15) == 0, YL_ERR_ARG, "boxes must be 16-byte aligned");
    YL_CHECK(workspace_bytes >= yl_nms_boxes_workspace_bytes(n), YL_ERR_WORKSPACE, "NMS workspace too small");
    char* ws = reinterpret_cast<char*>(workspace);
    uint32_t* cand_counts = reinterpret_cast<uint32_t*>(ws);
    unsigned long long* keys = reinterpret_cast<unsigned long long*>(ws + 256);
    float* kept_ws = reinterpret_cast<float*>(ws + 256 + yl::align_up((size_t)n * 8, 256));
    unsigned long long* kept_keys_ws = reinterpret_cast<unsigned long long*>(
        ws + 256 + yl::align_up((size_t)n * 8, 256) + yl::align_up((size_t)n * 5 * 4, 256));
    yl::nms_boxes_keys_kernel<<<yl::ceil_div(n, 256), 256, 0, s>>>(scores, n, keys, cand_counts);
    YL_LAUNCH_OK("nms_boxes_keys_kernel");

    yl::SelParams p;
    p.pred = boxes;
    p.nc = 1;
    p.A = n;
    p.lab_xywh = nullptr;
    p.lab_off = nullptr;
    p.cap = (unsigned long long)n;
    p.counts = cand_counts;
    p.keys = keys;
    p.thr = yl::thr_to_float(iou_thres);
    yl::thr_midpoint(p.thr, &p.thr_mid, &p.thr_tie_up);
    p.max_wh = 0.f;
    p.max_det = n;
    p.max_nms = n;
    p.kept_in_smem = 0;
    p.classwise = 0;
    p.dbg = yl::g_nms_dbg;
    p.kept_ws = kept_ws;
    p.kept_keys_ws = kept_keys_ws;
    p.out = nullptr;
    p.out_counts = count;
    p.keep = reinterpret_cast<long long*>(keep);
    const size_t smem = yl::sel_smem_bytes(0, false);
    YL_CHECK((int)smem <= yl::g_sel_max_smem, YL_ERR_UNSUPPORTED, "NMS needs %zu B shared memory (yl_init called?)",
             smem);
    yl::nms_select_kernel<1><<<1, yl::kSelThreads, smem, s>>>(p);
    YL_LAUNCH_OK("nms_select_kernel");
    return YL_OK;
}

int yl_xywh2xyxy_inplace(float* pred, int B, int C, int A, void* stream) {
    YL_CHECK(pred && B > 0 && C >= 4 && A > 0, YL_ERR_ARG, "bad arguments");
    const long long total = (long long)B * A;
    yl::xywh2xyxy_kernel<<<(unsigned)yl::ceil_div64(total, 256), 256, 0, (cudaStream_t)stream>>>(pred, C, A, total);
    YL_LAUNCH_OK("xywh2xyxy_kernel");
    return YL_OK;
}

int yl_scale_boxes(float* dets, const int32_t* counts, int B, int max_det, const float* params_dev, void* stream) {
    YL_CHECK(dets && counts && params_dev && B > 0 && max_det > 0, YL_ERR_ARG, "bad arguments");
    yl::scale_boxes_kernel<<<B, 128, 0, (cudaStream_t)stream>>>(dets, counts, max_det, params_dev);
    YL_LAUNCH_OK("scale_boxes_kernel");
    return YL_OK;
}

}  // extern "C"
