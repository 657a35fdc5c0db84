// COCO bbox evaluation on the GPU (the validator's `save_json=True`): pycocotools 2.0.x COCOeval.evaluate() and
// COCOeval.accumulate() for iouType="bbox", useCats=1 (the numpy restatement in the oracle package is the yardstick).
//
// evaluate (computeIoU + evaluateImg with maxDet = maxDets[-1]): one CTA per (category, image) pair that has a gt or a
// dt.  The pair's dts arrive in descending-score order (ties: input order, np.argsort(kind="mergesort")), already cut
// to maxDets[-1] by the host's grouping sort; they and the gts go to shared memory with, per area range, their `_ignore` flags and the stable
// "non-ignored first" order.  Each warp then runs whole (area, threshold) tasks: the dts are visited in rank order and
// the lanes scan the gts for the greedy match (see match_scan), so the only serial dimension is the dt order that the
// reference's greedy rule itself imposes.
//
// accumulate: one CTA per (category, area, maxDet, threshold).  The category's dt slots arrive contiguous, in the
// reference's concatenated order (descending score; ties by image rank, then rank within the image), gathered once
// after two stable device sorts, with the flags of each (area, threshold) in a row of their own.  tp / fp cumsums are exact integers; the precision envelope (`pr[i-1] = max(pr[i-1], pr[i])`) and
// np.searchsorted(rc, recThrs, "left") come out of one reverse pass: rc = tp / npig is monotone in tp, so the first
// index with rc >= recThr is the slot where tp first reaches c_r = min{c : c / npig >= recThr}.
//
// Compiled without fast-math; every fp64 operation is an explicit _rn intrinsic in the reference's order, so the
// results are bit-identical to numpy's.
#include "common.cuh"

namespace yl {
namespace {

constexpr int kEvalThreads = 256;
constexpr int kEvalWarps = kEvalThreads / 32;
constexpr int kAccThreads = 256;
constexpr int kAccWarps = kAccThreads / 32;
constexpr int kMaxAreas = 16;

__host__ __device__ inline size_t align8(size_t x) { return (x + 7) & ~size_t(7); }

// shared memory of one evaluate CTA for groups of at most G gts and D kept dts
__host__ __device__ inline size_t eval_smem_bytes(int G, int D, int A) {
    size_t b = align8((size_t)D * 5 * sizeof(double));          // dt x, y, w, h, area
    b += align8((size_t)D * sizeof(int64_t));                    // dt id
    b += align8((size_t)G * 5 * sizeof(double));                 // gt x, y, w, h, area
    b += align8((size_t)G * sizeof(int64_t));                    // gt id
    b += align8((size_t)A * G * sizeof(int32_t));                // per area: gt order (non-ignored first)
    b += align8((size_t)A * sizeof(int32_t));                    // per area: number of non-ignored gts
    b += align8((size_t)G);                                      // gt iscrowd
    b += align8((size_t)A * G);                                  // per area: gt _ignore
    b += align8((size_t)kEvalWarps * G);                         // per warp: gtm of its current task
    return b;
}

// maskApi bbIou for one (dt, gt) pair, in its operation order (boxes are x, y, w, h)
__device__ __forceinline__ double bb_iou(const double* d, const double* g, bool crowd) {
    const double w = __dsub_rn(fmin(__dadd_rn(d[2], d[0]), __dadd_rn(g[2], g[0])), fmax(d[0], g[0]));
    if (w <= 0.0) return 0.0;
    const double h = __dsub_rn(fmin(__dadd_rn(d[3], d[1]), __dadd_rn(g[3], g[1])), fmax(d[1], g[1]));
    if (h <= 0.0) return 0.0;
    const double i = __dmul_rn(w, h);
    const double da = __dmul_rn(d[2], d[3]);
    const double u = crowd ? da : __dsub_rn(__dadd_rn(da, __dmul_rn(g[2], g[3])), i);
    return __ddiv_rn(i, u);
}

// Ascending int64 key <=> descending score (-0.0 folded onto +0.0, which numpy's argsort treats as equal).
__device__ __forceinline__ long long desc_score_key(double s) {
    const unsigned long long b = (unsigned long long)__double_as_longlong(__dadd_rn(s, 0.0));
    const unsigned long long up = (b >> 63) ? ~b : (b | 0x8000000000000000ull);   // ascending with s, unsigned
    return (long long)(~up ^ 0x8000000000000000ull);
}

// One lane-parallel stretch of evaluateImg's gt loop: among gt positions [lo, hi) of the area's order that are not
// (matched and non-crowd) and have IoU >= thr, the highest IoU, equal IoU going to the LATER position (the reference
// updates `iou = ious[d, g]` and accepts `>=` afterwards).  Returns the winning position or -1, in every lane.
__device__ __forceinline__ int match_scan(int lo, int hi, const int32_t* ord, const double* dbox, const double* gbox,
                                          const uint8_t* crowd, const uint8_t* gtm, double thr, int lane) {
    double best = -1.0;
    int bpos = -1;
    for (int pos = lo + lane; pos < hi; pos += 32) {
        const int g = ord[pos];
        if (gtm[g] && !crowd[g]) continue;
        const double iou = bb_iou(dbox, gbox + (size_t)g * 4, crowd[g] != 0);
        if (iou >= thr && iou >= best) {
            best = iou;
            bpos = pos;
        }
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        const double ob = __shfl_xor_sync(0xffffffffu, best, off);
        const int op = __shfl_xor_sync(0xffffffffu, bpos, off);
        if (op >= 0 && (bpos < 0 || ob > best || (ob == best && op > bpos))) {
            best = ob;
            bpos = op;
        }
    }
    return bpos;
}

__global__ void __launch_bounds__(kEvalThreads) cocoeval_evaluate_kernel(yl_cocoeval_set s, yl_cocoeval_params prm,
                                                                         yl_cocoeval_slots out) {
    extern __shared__ __align__(16) unsigned char smem[];
    const int p = blockIdx.x;
    const int k = s.pair_cat[p];
    const int g0 = s.gt_off[p], G = s.gt_off[p + 1] - g0;
    const int s0 = s.slot_off[p], D = s.slot_off[p + 1] - s0;
    const size_t S = (size_t)s.n_slots;
    const int A = prm.A, T = prm.T;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

    unsigned char* q = smem;
    double* dbox = (double*)q;           q += align8((size_t)D * 4 * sizeof(double));
    double* darea = (double*)q;          q += align8((size_t)D * sizeof(double));
    int64_t* did = (int64_t*)q;          q += align8((size_t)D * sizeof(int64_t));
    double* gbox = (double*)q;           q += align8((size_t)G * 4 * sizeof(double));
    double* garea = (double*)q;          q += align8((size_t)G * sizeof(double));
    int64_t* gid = (int64_t*)q;          q += align8((size_t)G * sizeof(int64_t));
    int32_t* gorder = (int32_t*)q;       q += align8((size_t)A * G * sizeof(int32_t));
    int32_t* nonig = (int32_t*)q;        q += align8((size_t)A * sizeof(int32_t));
    uint8_t* crowd = (uint8_t*)q;        q += align8((size_t)G);
    uint8_t* gig = (uint8_t*)q;          q += align8((size_t)A * G);
    uint8_t* gtm_all = (uint8_t*)q;

    if (tid < A) nonig[tid] = 0;
    for (int g = tid; g < G; g += kEvalThreads) {
        for (int c = 0; c < 4; ++c) gbox[g * 4 + c] = s.gt_bbox[(size_t)(g0 + g) * 4 + c];
        garea[g] = s.gt_area[g0 + g];
        gid[g] = s.gt_id[g0 + g];
        crowd[g] = s.gt_iscrowd[g0 + g] ? 1 : 0;
    }
    // dts, already in rank order
    for (int d = tid; d < D; d += kEvalThreads) {
        for (int c = 0; c < 4; ++c) dbox[d * 4 + c] = s.dt_bbox[(size_t)(s0 + d) * 4 + c];
        darea[d] = s.dt_area[s0 + d];
        did[d] = s.dt_id[s0 + d];
        out.key[s0 + d] = desc_score_key(s.dt_score[s0 + d]);
        out.rank[s0 + d] = d;
    }
    __syncthreads();
    // per area range: gt._ignore = iscrowd || area < lo || area > hi (both bounds inclusive)
    for (int i = tid; i < A * G; i += kEvalThreads) {
        const int a = i / G, g = i - a * G;
        const double lo = prm.area_rng[2 * a], hi = prm.area_rng[2 * a + 1];
        gig[i] = (crowd[g] || garea[g] < lo || garea[g] > hi) ? 1 : 0;
    }
    __syncthreads();
    // np.argsort(_ignore, kind="mergesort"): non-ignored gts first, each part in file order
    for (int i = tid; i < A * G; i += kEvalThreads) {
        const int a = i / G, g = i - a * G;
        const uint8_t* ig = gig + a * G;
        int before_same = 0, n_keep = 0;
        for (int j = 0; j < G; ++j) {
            n_keep += ig[j] ? 0 : 1;
            before_same += (j < g && ig[j] == ig[g]) ? 1 : 0;
        }
        gorder[a * G + (ig[g] ? n_keep + before_same : before_same)] = g;
        if (g == 0) {
            nonig[a] = n_keep;
            atomicAdd(&out.npig[k * A + a], n_keep);
        }
    }
    __syncthreads();

    uint8_t* gtm = gtm_all + (size_t)warp * G;
    for (int task = warp; task < A * T; task += kEvalWarps) {
        const int a = task / T, t = task - a * T;
        const double lo = prm.area_rng[2 * a], hi = prm.area_rng[2 * a + 1];
        const double thr = fmin(prm.iou_thrs[t], 1.0 - 1e-10);
        const int32_t* ord = gorder + a * G;
        const int nk = nonig[a];
        for (int g = lane; g < G; g += 32) gtm[g] = 0;
        __syncwarp();
        for (int d = 0; d < D; ++d) {
            const double* db = dbox + d * 4;
            // a match among the non-ignored gts ends the loop at the first ignored one ("break" in evaluateImg)
            int pos = match_scan(0, nk, ord, db, gbox, crowd, gtm, thr, lane);
            if (pos < 0) pos = match_scan(nk, G, ord, db, gbox, crowd, gtm, thr, lane);
            if (lane == 0) {
                const int m = pos >= 0 ? ord[pos] : -1;
                const int64_t dtm = m >= 0 ? gid[m] : 0;   // a gt with id 0 leaves dtm = 0: "unmatched" downstream
                bool ig = m >= 0 && gig[a * G + m];
                if (m >= 0) gtm[m] = did[d] > 0 ? 1 : 0;    // gtm > 0 is the reference's "already matched"
                if (dtm == 0 && (darea[d] < lo || darea[d] > hi)) ig = true;
                out.flags[(size_t)(a * T + t) * S + s0 + d] = (uint8_t)((dtm != 0 ? 1 : 0) | (ig ? 2 : 0));
            }
            __syncwarp();
        }
        __syncwarp();
    }
}

// suffix (this lane and the lanes above it) inclusive scans of one warp
__device__ __forceinline__ int warp_suffix_sum(int v, int lane) {
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
        const int y = __shfl_down_sync(0xffffffffu, v, off);
        if (lane + off < 32) v += y;
    }
    return v;
}
__device__ __forceinline__ double warp_suffix_max(double v, int lane) {
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
        const double y = __shfl_down_sync(0xffffffffu, v, off);
        if (lane + off < 32) v = fmax(v, y);
    }
    return v;
}

__global__ void __launch_bounds__(kAccThreads) cocoeval_accumulate_kernel(yl_cocoeval_params prm, int K,
                                                                          int n_slots,
                                                                          const int32_t* __restrict__ cat_slot_off,
                                                                          const double* __restrict__ score,
                                                                          const int32_t* __restrict__ rank,
                                                                          const uint8_t* __restrict__ flags,
                                                                          const int32_t* __restrict__ npig_ka,
                                                                          double* precision, double* recall,
                                                                          double* scores) {
    extern __shared__ __align__(16) unsigned char smem[];
    const int A = prm.A, T = prm.T, M = prm.M, R = prm.R;
    int idx = blockIdx.x;
    const int t = idx % T; idx /= T;
    const int m = idx % M; idx /= M;
    const int a = idx % A;
    const int k = idx / A;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int max_det = prm.max_dets[m];
    const int c0 = cat_slot_off[k], n = cat_slot_off[k + 1] - c0;
    const int npig = npig_ka[k * A + a];
    const size_t rec_i = (((size_t)t * K + k) * A + a) * M + m;
    auto out_i = [&](int r) { return ((((size_t)t * R + r) * K + k) * A + a) * M + m; };
    if (npig == 0) {   // no non-ignored gt in this category: precision / recall / scores keep -1
        for (int r = tid; r < R; r += kAccThreads) {
            precision[out_i(r)] = -1.0;
            scores[out_i(r)] = -1.0;
        }
        if (tid == 0) recall[rec_i] = -1.0;
        return;
    }
    double* qv = (double*)smem;
    double* sv = qv + R;
    int* cr = (int*)(sv + R);
    __shared__ int red_i[3][kAccWarps];
    __shared__ double red_d[kAccWarps];
    const double dnp = (double)npig;
    for (int r = tid; r < R; r += kAccThreads) {
        qv[r] = 0.0;
        sv[r] = 0.0;
        // c_r = min{c in [0, npig] : c / npig >= recThrs[r]} (INT_MAX: never reached)
        const double thr = prm.rec_thrs[r];
        const double c_est = ceil(thr * dnp);
        long long c = c_est > 0.0 ? (c_est < dnp ? (long long)c_est : npig) : 0;
        while (c > 0 && __ddiv_rn((double)(c - 1), dnp) >= thr) --c;
        while (c <= npig && !(__ddiv_rn((double)c, dnp) >= thr)) ++c;
        cr[r] = c > npig ? 0x7fffffff : (int)c;
    }
    const uint8_t* fl = flags + (size_t)(a * T + t) * n_slots;
    auto load = [&](int j, bool& sel, int& tp, int& fp, size_t& slot) {
        slot = (size_t)c0 + j;
        sel = rank[slot] < max_det;
        const uint8_t f = fl[slot];
        tp = (sel && f == 1) ? 1 : 0;   // matched and not ignored
        fp = (sel && f == 0) ? 1 : 0;   // unmatched and not ignored
    };
    // pass 1: totals and the first kept slot
    int tp_tot = 0, fp_tot = 0, first = 0x7fffffff;
    for (int j = tid; j < n; j += kAccThreads) {
        bool sel;
        int tp, fp;
        size_t slot;
        load(j, sel, tp, fp, slot);
        tp_tot += tp;
        fp_tot += fp;
        if (sel && j < first) first = j;
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        tp_tot += __shfl_xor_sync(0xffffffffu, tp_tot, off);
        fp_tot += __shfl_xor_sync(0xffffffffu, fp_tot, off);
        first = min(first, __shfl_xor_sync(0xffffffffu, first, off));
    }
    if (lane == 0) {
        red_i[0][warp] = tp_tot;
        red_i[1][warp] = fp_tot;
        red_i[2][warp] = first;
    }
    __syncthreads();
    tp_tot = fp_tot = 0;
    first = 0x7fffffff;
    for (int w = 0; w < kAccWarps; ++w) {
        tp_tot += red_i[0][w];
        fp_tot += red_i[1][w];
        first = min(first, red_i[2][w]);
    }
    if (tid == 0) recall[rec_i] = first < n ? __ddiv_rn((double)tp_tot, dnp) : 0.0;
    __syncthreads();

    // pass 2: chunks from the last to the first; cumulative tp / fp at j = totals minus the counts after j
    int after_tp = 0, after_fp = 0;
    double after_max = -1.0;
    const double eps = 2.220446049250313e-16;   // np.spacing(1)
    for (int base = ((n - 1) / kAccThreads) * kAccThreads; base >= 0 && n > 0; base -= kAccThreads) {
        const int j = base + tid;
        bool sel = false;
        int tp = 0, fp = 0;
        size_t slot = 0;
        if (j < n) load(j, sel, tp, fp, slot);
        const int stp = warp_suffix_sum(tp, lane), sfp = warp_suffix_sum(fp, lane);
        if (lane == 0) {
            red_i[0][warp] = stp;
            red_i[1][warp] = sfp;
        }
        __syncthreads();
        int up_tp = 0, up_fp = 0, ch_tp = 0, ch_fp = 0;
        for (int w = 0; w < kAccWarps; ++w) {
            if (w > warp) {
                up_tp += red_i[0][w];
                up_fp += red_i[1][w];
            }
            ch_tp += red_i[0][w];
            ch_fp += red_i[1][w];
        }
        const int tpc = tp_tot - (after_tp + up_tp + stp - tp);
        const int fpc = fp_tot - (after_fp + up_fp + sfp - fp);
        const double dtp = (double)tpc;
        const double pr = sel ? __ddiv_rn(dtp, __dadd_rn(__dadd_rn((double)fpc, dtp), eps)) : -1.0;
        const double smax = warp_suffix_max(pr, lane);
        if (lane == 0) red_d[warp] = smax;
        __syncthreads();
        double env = fmax(smax, after_max), ch_max = after_max;
        for (int w = 0; w < kAccWarps; ++w) {
            if (w > warp) env = fmax(env, red_d[w]);
            ch_max = fmax(ch_max, red_d[w]);
        }
        if (sel && (j == first || tp)) {
            const double sc = score[slot];
            for (int r = 0; r < R; ++r)
                if (j == first ? cr[r] <= tpc : cr[r] == tpc) {
                    qv[r] = env;
                    sv[r] = sc;
                }
        }
        after_tp += ch_tp;
        after_fp += ch_fp;
        after_max = ch_max;
        __syncthreads();
    }
    __syncthreads();
    for (int r = tid; r < R; r += kAccThreads) {
        precision[out_i(r)] = qv[r];
        scores[out_i(r)] = sv[r];
    }
}

}  // namespace
}  // namespace yl

using namespace yl;

extern "C" {

int yl_cocoeval_evaluate(const yl_cocoeval_set* set, const yl_cocoeval_params* prm, const yl_cocoeval_slots* out,
                         void* stream) {
    YL_CHECK(set && prm && out, 1, "yl_cocoeval_evaluate: null argument");
    YL_CHECK(prm->A >= 1 && prm->A <= kMaxAreas && prm->T >= 1 && prm->R >= 1 && prm->M >= 1, 1,
             "yl_cocoeval_evaluate: bad parameter counts (T=%d R=%d A=%d M=%d)", prm->T, prm->R, prm->A, prm->M);
    YL_CHECK(set->n_pairs >= 0 && set->n_cats >= 0 && set->n_slots >= 0 && set->max_gt >= 0 && set->max_dt >= 0, 1,
             "yl_cocoeval_evaluate: negative sizes");
    cudaStream_t st = (cudaStream_t)stream;
    if (set->n_cats > 0) YL_CUDA(cudaMemsetAsync(out->npig, 0, (size_t)set->n_cats * prm->A * sizeof(int32_t), st));
    if (set->n_pairs == 0) return 0;
    const size_t smem = eval_smem_bytes(set->max_gt, set->max_dt, prm->A);
    int dev = 0, optin = 0;
    YL_CUDA(cudaGetDevice(&dev));
    YL_CUDA(cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
    YL_CHECK(smem <= (size_t)optin, 1,
             "yl_cocoeval_evaluate: %d gts / %d dts in one (image, category) need %zu bytes of shared memory (max %d)",
             set->max_gt, set->max_dt, smem, optin);
    if (smem > 48 * 1024)
        YL_CUDA(cudaFuncSetAttribute(cocoeval_evaluate_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    cocoeval_evaluate_kernel<<<set->n_pairs, kEvalThreads, smem, st>>>(*set, *prm, *out);
    YL_LAUNCH_OK("cocoeval_evaluate_kernel");
    return 0;
}

int yl_cocoeval_accumulate(const yl_cocoeval_params* prm, int n_cats, int n_slots, const int32_t* cat_slot_off,
                           const double* score, const int32_t* rank, const uint8_t* flags, const int32_t* npig,
                           double* precision, double* recall, double* scores, void* stream) {
    YL_CHECK(prm && cat_slot_off && npig && precision && recall && scores && n_slots >= 0, 1,
             "yl_cocoeval_accumulate: null argument");
    YL_CHECK(prm->A >= 1 && prm->T >= 1 && prm->R >= 1 && prm->M >= 1 && n_cats >= 0, 1,
             "yl_cocoeval_accumulate: bad parameter counts");
    const long long grid = (long long)n_cats * prm->A * prm->M * prm->T;
    YL_CHECK(grid < 0x7fffffffLL, 1, "yl_cocoeval_accumulate: too many (category, area, maxDet, threshold) cells");
    if (grid == 0) return 0;
    const size_t smem = (size_t)prm->R * (2 * sizeof(double) + sizeof(int));
    YL_CHECK(smem <= 48 * 1024, 1, "yl_cocoeval_accumulate: %d recall thresholds is too many", prm->R);
    cocoeval_accumulate_kernel<<<(unsigned)grid, kAccThreads, smem, (cudaStream_t)stream>>>(
        *prm, n_cats, n_slots, cat_slot_off, score, rank, flags, npig, precision, recall, scores);
    YL_LAUNCH_OK("cocoeval_accumulate_kernel");
    return 0;
}

}  // extern "C"
