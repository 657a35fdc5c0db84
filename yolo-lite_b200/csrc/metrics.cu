// Validator metric on the GPU (SURVEY §8f rank 4): box_iou + match_predictions for a whole batch in one launch.
//
//   reference: utils/metrics.py:51-70 (box_iou, fp32, eps = 1e-7), engine/validator.py:410-429 (_process_batch)
//              and :195-233 (match_predictions, the non-scipy branch), looped per image in update_metrics :313-360.
//
// match_predictions, restated: for one IoU threshold, among all (label, detection) pairs of the same class with
// IoU >= threshold, (1) every detection keeps only its highest-IoU label, (2) every label keeps only the
// LOWEST-INDEX detection that chose it (np.unique returns first occurrences of the index-sorted rows, and the
// detections arrive sorted by confidence).  A detection's best label does not depend on the threshold, so one
// pass over the labels per detection serves all thresholds.
// Compiled without fast-math; the IoU uses explicit _rn intrinsics in the reference's operation order so the
// comparisons against the thresholds see the same fp32 values as the CPU path (exact IoU ties between two labels
// of one detection are resolved towards the lower label index; numpy's order is unspecified there).
//
// ConfusionMatrix.process_batch (the validator's `plots=True`), restated: detections with conf > the matrix's conf
// are paired with labels of ANY class at IoU > iou_thres (strict); every detection keeps its highest-IoU pair, then
// every label keeps the highest-IoU pair among those that remain (upstream re-sorts by IoU before the second
// np.unique).  Exact IoU ties go to the lower label index, then to the lower detection index (upstream's order comes
// from np.argsort and is unspecified there).  A matched label counts at [cls(det), cls(gt)], an unmatched label at
// [nc, cls(gt)], a kept detection in no surviving pair at [cls(det), nc].
#include "common.cuh"

namespace yl {

constexpr int kMaxThr = 16;

// box_iou(gt, det) of one pair: inter / (area_gt + area_det - inter + eps), left to right, each op rounded
__device__ __forceinline__ float iou_gt_det(const float* g, float x1, float y1, float x2, float y2, float area_d,
                                            float eps) {
    const float iw = fmaxf(__fsub_rn(fminf(g[2], x2), fmaxf(g[0], x1)), 0.f);
    const float ih = fmaxf(__fsub_rn(fminf(g[3], y2), fmaxf(g[1], y1)), 0.f);
    const float inter = __fmul_rn(iw, ih);
    const float area_g = __fmul_rn(__fsub_rn(g[2], g[0]), __fsub_rn(g[3], g[1]));
    return __fdiv_rn(inter, __fadd_rn(__fsub_rn(__fadd_rn(area_g, area_d), inter), eps));
}

__global__ void __launch_bounds__(256) match_predictions_kernel(const float* __restrict__ dets, const int32_t* __restrict__ counts,
                                                                int max_det, const float* __restrict__ gt_boxes,
                                                                const float* __restrict__ gt_cls,
                                                                const int32_t* __restrict__ gt_offsets,
                                                                const float* __restrict__ thr, int nthr, float eps,
                                                                uint8_t* __restrict__ tp) {
    extern __shared__ int32_t win[];   // [nthr][L]: lowest detection index that matched label l at threshold t; then [D]: best label of d
    const int b = blockIdx.x;
    const int l0 = gt_offsets[b], L = gt_offsets[b + 1] - l0;
    const int D = min(counts[b], max_det);
    for (int i = threadIdx.x; i < nthr * L; i += blockDim.x) win[i] = 0x7fffffff;
    __syncthreads();
    float th[kMaxThr];
#pragma unroll
    for (int t = 0; t < kMaxThr; ++t) th[t] = t < nthr ? thr[t] : 2.f;
    // detections are processed in rounds of blockDim; each thread remembers its detection's best label
    for (int d0 = 0; d0 < D; d0 += blockDim.x) {
        const int d = d0 + threadIdx.x;
        float best = 0.f;
        int bl = -1;
        if (d < D) {
            const float* p = dets + ((long long)b * max_det + d) * 6;
            const float x1 = p[0], y1 = p[1], x2 = p[2], y2 = p[3], pc = p[5];
            const float area_d = __fmul_rn(__fsub_rn(x2, x1), __fsub_rn(y2, y1));
            for (int l = 0; l < L; ++l) {
                const float* g = gt_boxes + (long long)(l0 + l) * 4;
                if (gt_cls[l0 + l] != pc) continue;                    // iou * correct_class
                const float iou = iou_gt_det(g, x1, y1, x2, y2, area_d, eps);
                if (iou > best) {
                    best = iou;
                    bl = l;
                }
            }
            if (bl >= 0)
                for (int t = 0; t < nthr; ++t)
                    if (best >= th[t]) atomicMin(&win[t * L + bl], d);
        }
        // the winners are only final once every detection has voted: keep this detection's candidate flags (in tp)
        // and its label (side array behind the winners) for the resolve pass below
        if (d < D) {
            uint8_t* o = tp + ((long long)b * max_det + d) * nthr;
            for (int t = 0; t < nthr; ++t) o[t] = (bl >= 0 && best >= th[t]) ? (uint8_t)1 : (uint8_t)0;
            win[nthr * L + d] = bl;
        }
    }
    __syncthreads();
    for (int d = threadIdx.x; d < D; d += blockDim.x) {
        const int bl = win[nthr * L + d];
        uint8_t* o = tp + ((long long)b * max_det + d) * nthr;
        for (int t = 0; t < nthr; ++t) o[t] = (o[t] && bl >= 0 && win[t * L + bl] == d) ? (uint8_t)1 : (uint8_t)0;
    }
    // rows beyond the image's detection count are defined as all-false
    for (int i = D * nthr + threadIdx.x; i < max_det * nthr; i += blockDim.x) tp[(long long)b * max_det * nthr + i] = 0;
}

__device__ __forceinline__ void cm_add(unsigned long long* matrix, int nc, int pc, int gc) {
    const bool ok = pc >= 0 && pc <= nc && gc >= 0 && gc <= nc;
    atomicAdd(matrix + (ok ? (long long)pc * (nc + 1) + gc : (long long)(nc + 1) * (nc + 1)), 1ull);
}

__global__ void __launch_bounds__(256) confusion_matrix_kernel(const float* __restrict__ dets,
                                                               const int32_t* __restrict__ counts, int max_det,
                                                               const float* __restrict__ gt_boxes,
                                                               const float* __restrict__ gt_cls,
                                                               const int32_t* __restrict__ gt_offsets, int nc, float conf,
                                                               float iou_thres, float eps,
                                                               unsigned long long* __restrict__ matrix) {
    // [L]: best (IoU bits << 32 | ~d) among the detections whose best pair is label l (0: none); then [D]: best label
    // of detection d (-1: no pair above iou_thres, -2: conf filtered)
    extern __shared__ unsigned long long cwin[];
    const int b = blockIdx.x;
    const int l0 = gt_offsets[b], L = gt_offsets[b + 1] - l0;
    const int D = min(counts[b], max_det);
    int* dlab = reinterpret_cast<int*>(cwin + L);
    for (int i = threadIdx.x; i < L; i += blockDim.x) cwin[i] = 0ull;
    __syncthreads();
    for (int d = threadIdx.x; d < D; d += blockDim.x) {
        const float* p = dets + ((long long)b * max_det + d) * 6;
        int bl = -2;
        if (p[4] > conf) {
            const float x1 = p[0], y1 = p[1], x2 = p[2], y2 = p[3];
            const float area_d = __fmul_rn(__fsub_rn(x2, x1), __fsub_rn(y2, y1));
            float best = iou_thres;   // strict: a pair exactly at the threshold is no candidate
            bl = -1;
            for (int l = 0; l < L; ++l) {
                const float iou = iou_gt_det(gt_boxes + (long long)(l0 + l) * 4, x1, y1, x2, y2, area_d, eps);
                if (iou > best) {     // strict: ties keep the lower label index
                    best = iou;
                    bl = l;
                }
            }
            // IoU > iou_thres >= 0, so its bits order like its value; ~d prefers the lower detection index on ties
            if (bl >= 0) atomicMax(&cwin[bl], ((unsigned long long)__float_as_uint(best) << 32) | (uint32_t)~(uint32_t)d);
        }
        dlab[d] = bl;
    }
    __syncthreads();
    for (int l = threadIdx.x; l < L; l += blockDim.x) {
        const unsigned long long w = cwin[l];
        int pc = nc;
        if (w) pc = (int)dets[((long long)b * max_det + (int)~(uint32_t)(w & 0xffffffffull)) * 6 + 5];
        cm_add(matrix, nc, pc, (int)gt_cls[l0 + l]);
    }
    for (int d = threadIdx.x; d < D; d += blockDim.x) {
        const int bl = dlab[d];
        if (bl == -2) continue;
        if (bl >= 0 && (uint32_t)(cwin[bl] & 0xffffffffull) == ~(uint32_t)d) continue;   // matched
        cm_add(matrix, nc, (int)dets[((long long)b * max_det + d) * 6 + 5], nc);
    }
}

// per-device setup (called by yl_init): crowded images need more than the default 48 KB of dynamic shared memory
int init_metrics() {
    YL_CUDA(cudaFuncSetAttribute(match_predictions_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    YL_CUDA(cudaFuncSetAttribute(confusion_matrix_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    return YL_OK;
}

}  // namespace yl

extern "C" int yl_match_predictions(const float* dets, const int32_t* counts, int B, int max_det, const float* gt_boxes,
                                    const float* gt_cls, const int32_t* gt_offsets, int max_labels_per_image,
                                    const float* iou_thresholds_dev, int n_thresholds, uint8_t* tp, void* stream) {
    YL_CHECK(dets && counts && gt_offsets && iou_thresholds_dev && tp, YL_ERR_ARG, "null pointer");
    YL_CHECK(B >= 1 && max_det >= 1 && n_thresholds >= 1 && n_thresholds <= yl::kMaxThr, YL_ERR_ARG, "bad match dims");
    YL_CHECK(max_labels_per_image >= 0, YL_ERR_ARG, "bad label count");
    const size_t smem = ((size_t)n_thresholds * max_labels_per_image + max_det) * sizeof(int32_t);
    YL_CHECK(smem <= 200 * 1024, YL_ERR_UNSUPPORTED, "too many labels per image for the matching kernel (%d)", max_labels_per_image);
    yl::match_predictions_kernel<<<B, 256, smem, (cudaStream_t)stream>>>(dets, counts, max_det, gt_boxes, gt_cls, gt_offsets,
                                                                         iou_thresholds_dev, n_thresholds, 1e-7f, tp);
    YL_LAUNCH_OK("match_predictions_kernel");
    return YL_OK;
}

extern "C" int yl_confusion_matrix(const float* dets, const int32_t* counts, int B, int max_det, const float* gt_boxes,
                                   const float* gt_cls, const int32_t* gt_offsets, int max_labels_per_image, int nc,
                                   float conf, float iou_thres, int64_t* matrix, void* stream) {
    YL_CHECK(dets && counts && gt_offsets && matrix, YL_ERR_ARG, "null pointer");
    YL_CHECK(B >= 1 && max_det >= 1 && nc >= 1, YL_ERR_ARG, "bad confusion matrix dims");
    YL_CHECK(max_labels_per_image >= 0 && (max_labels_per_image == 0 || (gt_boxes && gt_cls)), YL_ERR_ARG,
             "bad labels");
    YL_CHECK(iou_thres >= 0.f && iou_thres <= 1.f, YL_ERR_ARG, "iou_thres must be in [0,1]");
    const size_t smem = (size_t)max_labels_per_image * 8 + (size_t)max_det * 4;
    YL_CHECK(smem <= 200 * 1024, YL_ERR_UNSUPPORTED, "too many labels per image for the confusion kernel (%d)",
             max_labels_per_image);
    yl::confusion_matrix_kernel<<<B, 256, smem, (cudaStream_t)stream>>>(dets, counts, max_det, gt_boxes, gt_cls,
                                                                         gt_offsets, nc, conf, iou_thres, 1e-7f,
                                                                         reinterpret_cast<unsigned long long*>(matrix));
    YL_LAUNCH_OK("confusion_matrix_kernel");
    return YL_OK;
}
