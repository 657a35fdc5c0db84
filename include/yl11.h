/* yl11.h — C-ABI of libyl11.so: the B200 (sm_100a) kernels behind the YOLO11 inference path of YOLO-Lite.
 *
 * The reference (dongyunjinyu/YOLO-Lite) is pure Python and has no FFI; every entry point below replaces a
 * *library call site* of the reference (ATen / cuDNN / torchvision), cited as `file:line` relative to the
 * reference root.  The reference-side binding is a ctypes stub (see INTEGRATION.md); the shipped binding is
 * yolo-lite_b200/yololite/_C.py.
 *
 * Conventions
 *   - plain pointers + sizes only; all pointers are DEVICE pointers unless stated otherwise;
 *   - every call is asynchronous on the caller's `stream` (a cudaStream_t passed as void*), never allocates,
 *     never synchronises, and is CUDA-graph capturable;
 *   - return 0 on success, negative yl_status on failure; yl_last_error_string() gives the text
 *     (thread-local);
 *   - activations are NHWC ("pixel major") bf16; a yl_tensor is a channel slice [coff, coff+c) of a buffer
 *     with `cstride` channels per pixel, so channel-concat is aliasing, not a copy.
 */
#ifndef YL11_H
#define YL11_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define YL11_VERSION 200

typedef enum yl_status {
    YL_OK = 0,
    YL_ERR_ARG = -1,       /* bad shape / alignment / null pointer            */
    YL_ERR_CUDA = -2,      /* a CUDA runtime / driver call failed             */
    YL_ERR_UNSUPPORTED = -3,
    YL_ERR_WORKSPACE = -4, /* workspace too small                              */
    YL_ERR_NO_DEVICE = -5  /* no sm_100 device: the library has no CPU path    */
} yl_status;

/* YL_U8 / YL_F16 are image-ingest types only (the caller's batch); activations are bf16, head outputs f32 */
typedef enum yl_dtype { YL_BF16 = 0, YL_F32 = 1, YL_U8 = 2, YL_F16 = 3 } yl_dtype;
typedef enum yl_act { YL_ACT_NONE = 0, YL_ACT_SILU = 1 } yl_act;
typedef enum yl_conv_impl { YL_IMPL_AUTO = 0, YL_IMPL_DIRECT = 1, YL_IMPL_TCGEN05 = 2 } yl_conv_impl;

/* NHWC view: element (n,h,w,ch) lives at data[((n*h_dim + h)*w_dim + w)*cstride + coff + ch]. */
typedef struct yl_tensor {
    void* data;
    int32_t n, h, w, c;
    int32_t cstride; /* channels per pixel of the underlying buffer (>= coff + c) */
    int32_t coff;    /* first channel of the slice                               */
    int32_t dtype;   /* yl_dtype                                                  */
    int32_t _pad;
} yl_tensor;

/* ---- runtime ------------------------------------------------------------------------------------------- */
int yl_version(void);
const char* yl_last_error_string(void);
/* Bind to `device`, check it is sm_100, resolve the TMA encoder and opt kernels into large shared memory.
 * Must be called once per process before any other entry point. */
int yl_init(int device);
/* Programmatic dependent launch: by default every kernel of the library is launched with the programmatic
 * stream-serialization attribute (its prologue may overlap the previous kernel of the stream; it executes
 * griddepcontrol.wait before touching activations).  yl_set_pdl(0) makes subsequent launches plain (used for a
 * launch that follows a cross-stream event wait); returns the previous setting.  The setting belongs to the CALLING
 * THREAD (thread-local, like the CUDA current device): other threads' launches are unaffected. */
int yl_set_pdl(int enabled);
/* Debug aid: the next `capacity` tcgen05 conv launches record 8 %globaltimer stamps (ns) of CTA 0 into
 * device_buf[launch][8]: start, prologue done, dependency wait done, first operands landed, first accumulator
 * ready, last store issued, staging drained, exit.  NULL disables.  Arms the calling thread's launches only
 * (thread-local); a separate instantiation of the kernel carries the stamps, production launches never pay for them. */
int yl_debug_timeline(unsigned long long* device_buf, int capacity);

/* ---- weight preparation (one-time) ----------------------------------------------------------------------
 * Replaces the fold the reference never performs at inference (utils/torch_utils.py:182-209 is the formula:
 * w' = w * gamma / sqrt(var + eps), b' = beta - mean * gamma / sqrt(var + eps) [+ conv bias scaled]).
 * Dense: w_oihw [co][ci][k][k] fp32 -> packed bf16 [co_pad][k*k][ci_pad] (tap-major, channel-minor = the
 * K order of the implicit GEMM).  Depthwise (ci == 1, depthwise != 0): -> bf16 [k*k][co_pad].
 * gamma/beta/mean/var may all be NULL (plain nn.Conv2d, head.py:39,48); conv_bias may be NULL. */
int yl_fold_bn_pack(const float* w_oihw, const float* gamma, const float* beta, const float* mean,
                    const float* var, const float* conv_bias, float eps, int co, int ci, int k, int co_pad,
                    int ci_pad, int depthwise, void* w_packed, float* bias_out, void* stream);

/* ---- layout ------------------------------------------------------------------------------------------- */
/* predictor.py:81-84 (`.to(device).float()`): NCHW fp32 image batch -> NHWC bf16 slice. */
int yl_nchw_to_nhwc(const float* x_nchw, const yl_tensor* y, void* stream);
/* NHWC slice (bf16 or f32) -> dense NCHW fp32 (module-level API returns reference-layout tensors). */
int yl_nhwc_to_nchw(const yl_tensor* x, float* y_nchw, void* stream);
/* conv.py:321-331 Concat fallback when aliasing is impossible: copy a channel slice into another. */
int yl_copy_slice(const yl_tensor* x, const yl_tensor* y, void* stream);
/* nn.Upsample(None, 2, "nearest") (cfg/yolo11.yaml:31,35): y is (n, 2h, 2w, c). */
int yl_upsample2x(const yl_tensor* x, const yl_tensor* y, void* stream);

/* ---- convolution ---------------------------------------------------------------------------------------
 * Replaces Conv.forward = act(bn(conv(x))) (nn/modules/conv.py:35-53), Bottleneck's residual add
 * (block.py:343), the PSABlock adds (block.py:951-952) and the torch.cat that follows a conv
 * (block.py:233-235, 259, 184) via the output slice.  Dense k in {1,3}, stride in {1,2}, pad = k/2.
 *   y = [res +] act(conv(x, w) + bias)
 * `y.h/y.w` are the conv output dims; with upsample2x != 0 each result pixel is replicated into the 2x2
 * block of a (n, 2h, 2w) buffer described by `y` (then y.h/y.w are the *upsampled* dims).
 * The tcgen05 path stores through TMA: out-of-range rows/channels are clipped by the tensor map. */
/* Optional Detect-decode epilogue of a 1x1 head conv (head.py:95-126 fused into the conv that produces the
 * logits, so the raw head map need not be written and re-read): the conv result (+bias, no activation) of
 * pixel (b, a_local) is decoded straight into the prediction tensor pred (B, 4+nc, A) fp32:
 *   mode YL_DET_BOX  (co == 4*reg_max, reg_max == 16): DFL softmax-expectation per side (block.py:51-69),
 *        dist2bbox around the anchor centre (tal.py:341-350), * stride  -> pred[b, 0:4, anchor0 + a_local]
 *   mode YL_DET_CLS  (co == nc): sigmoid                               -> pred[b, 4:4+nc, anchor0 + a_local]
 *   mode YL_DET_CLS_FILTER (co == nc): sigmoid, best class per anchor and the confidence test of
 *        ops.non_max_suppression (utils/ops.py:203, 242-244: `conf, j = cls.max(1)`, strict `conf > conf_thres`, ties
 *        keep the lowest class index), all in the conv epilogue: every passing anchor becomes one candidate key in
 *        the NMS workspace `cand_ws` (layout of yl_nms_workspace_bytes(B, A, nc, 0), counters zeroed by
 *        yl_nms_begin), exactly the key yl_nms_batched's filter kernel would emit from the stored scores.  The class
 *        rows of pred are then never written (nor re-read): yl_nms_select finishes the step.  Single-label NMS only.
 * With det.pred != NULL the NHWC destination `y` becomes optional (y.data may be NULL: no raw map at all). */
typedef enum yl_det_mode { YL_DET_NONE = 0, YL_DET_BOX = 1, YL_DET_CLS = 2, YL_DET_CLS_FILTER = 3 } yl_det_mode;
typedef struct yl_det_epilogue {
    float* pred;     /* NULL: plain conv epilogue */
    int32_t mode;    /* yl_det_mode */
    int32_t reg_max; /* 16 */
    int32_t nc;      /* classes: pred has 4 + nc rows */
    int32_t A;       /* anchors per image over all levels */
    int32_t anchor0; /* first anchor of this level */
    float stride;    /* level stride in pixels */
    float conf;      /* YL_DET_CLS_FILTER: confidence threshold */
    int32_t _pad;
    void* cand_ws;   /* YL_DET_CLS_FILTER: NMS workspace receiving the candidates */
} yl_det_epilogue;

typedef struct yl_conv_args {
    yl_tensor x;
    yl_tensor y;   /* bf16 or f32 */
    yl_tensor res; /* res.data == NULL: no residual; else same dims as the conv output, bf16 */
    yl_tensor y_up; /* y_up.data == NULL: none; else a second destination (n, 2h, 2w) of y's dtype that
                       receives the result replicated 2x2: a conv output that feeds both a Concat and an
                       nn.Upsample -> Concat (cfg/yolo11.yaml:31-44) is stored once per consumer        */
    const void* w; /* packed by yl_fold_bn_pack                                              */
    const float* bias;
    int32_t k, stride;
    int32_t ci_pad, co_pad; /* packed weight dims; x.c <= ci_pad, y.c <= co_pad             */
    int32_t act;            /* yl_act                                                         */
    int32_t upsample2x;
    int32_t impl;           /* yl_conv_impl                                                   */
    int32_t _pad;
    yl_det_epilogue det;    /* det.pred == NULL: none (tcgen05 path only, k = 1, stride 1, no act/res) */
} yl_conv_args;
int yl_conv_bn_act(const yl_conv_args* a, void* stream);
/* Back-to-back form for the tail of a Detect BOX branch on the engine path (head.py:39-41, 59-65): the branch's last
 * Conv(c2, c2, 3) and the final nn.Conv2d(c2, 4 * reg_max, 1) with its DFL / dist2bbox decode in ONE launch.  `conv` is the
 * 3x3 conv (k in {1,3}, y.data == NULL: its result is not stored, y gives dims / channels <= 128); its epilogue rounds the
 * result to bf16 into swizzled shared-memory tiles that are the A operand of a second tcgen05 GEMM with `head`'s weights
 * (head: 1x1, no activation, y.data == NULL, det.mode = YL_DET_BOX or YL_DET_CLS, its x is ignored).  Bit-identical to
 * yl_conv_bn_act(conv) followed by yl_conv_bn_act(head). */
int yl_conv_b2b_det_supported(const yl_conv_args* conv, const yl_conv_args* head);
int yl_conv_b2b_det(const yl_conv_args* conv, const yl_conv_args* head, void* stream);
/* 1 if the tcgen05 implicit-GEMM path can run this problem, 0 if it needs the direct kernel. */
int yl_conv_tc_supported(const yl_conv_args* a);
/* How the tcgen05 path would run this problem (the host-side dispatch of conv_tc.cu; nothing is launched): tests
 * assert through it that the batch-size-dependent paths (image-stacked tiles, N split, halo patch, resident weights)
 * are the ones a parity case exercised. */
typedef struct yl_conv_tc_plan {
    int flat;               /* 1x1: the (n,h,w) extent is one axis, tiles are 128 consecutive pixels */
    int patch;              /* 3x3 s1 thin input: one halo-patch TMA box per tile, resident 9-tap weights */
    int wres;               /* all weight tiles resident in shared memory (ring carries activations only) */
    int tile_w, tile_h, tile_n;   /* A-tile box; tile_n > 1 = the same window of consecutive images stacked */
    int m_tiles, n_tiles;   /* n_tiles == 2 with co <= 256: the wave-quantisation N split */
    int co_tile, kblk, stages, grid, smem_bytes, tmem_cols;
    int cw;                 /* TMEM columns per epilogue chunk (16 or 32) */
    int stg_sub;            /* chunks per staged TMA store (2: 128-byte bf16 pixel rows) */
    int epi_kind;           /* epilogue instantiation: 0-3 bf16 (SiLU?, residual?), 4 / 5 / 6 Detect box / class /
                               class filter, 7 generic (f32 out, 16-column chunks, stored Detect raw map) */
} yl_conv_tc_plan;
int yl_conv_tc_info(const yl_conv_args* a, yl_conv_tc_plan* out);

/* A chain of convolution layers in ONE launch (csrc/conv_chain.cu): the consecutive Conv modules of the small feature
 * maps — the C3k / Bottleneck chains, SPPF and C2PSA 1x1 convs of nn/tasks.py:118-145's layer loop (block.py:165-184,
 * 330-343, 720-739, 999-1038) — each of which is a launch-latency chain rather than work when run as its own kernel.
 * One thread-block cluster (4 CTAs) owns one image for the whole chain; layers hand over through L2 and a cluster
 * barrier.  Every layer is a yl_conv_args of the bf16 -> bf16 kind (k in {1,3}, stride in {1,2}, optional SiLU /
 * residual / 2x-upsampled second destination; no Detect epilogue), all with the same batch; a layer may read anything
 * earlier layers of the chain (or earlier launches) wrote.  Results are bit-identical to the layers launched one by one.
 *   yl_conv_chain_build plans the layers and fills `desc_dev` (device, >= yl_conv_chain_desc_bytes(n), 128-byte aligned,
 *   owned by the caller, must outlive the chain); it synchronises `stream` once.  yl_conv_chain_run is asynchronous and
 *   graph-capturable like every other launch. */
typedef struct yl_conv_chain {
    void* desc;
    int32_t n_layers, batch, cluster, smem_bytes, tmem_cols, reserved;
} yl_conv_chain;
size_t yl_conv_chain_desc_bytes(int n_layers);
/* 1 if this layer can be a member of a chain */
int yl_conv_chain_supported(const yl_conv_args* a);
int yl_conv_chain_build(const yl_conv_args* layers, int n_layers, void* desc_dev, size_t desc_bytes, yl_conv_chain* out,
                        void* stream);
int yl_conv_chain_run(const yl_conv_chain* chain, void* stream);
/* Debug aid (tools/chain_timeline.py): chain launches of the calling thread record, per layer, 6 %globaltimer stamps (ns)
 * of CTA 0 into device_buf[layer][8]: layer start, first operands landed, last MMA issued, epilogue entered, epilogue
 * returned (stores complete), cluster barrier passed.  NULL disables. */
int yl_conv_chain_debug(unsigned long long* device_buf);

/* First layer fused with the image ingest (predictor.py:81-84 + conv.py:35-53): reads the NCHW fp32 batch
 * (values rounded to bf16 like every other activation), 3x3 stride-2 pad-1 conv, <= 4 input channels, folded
 * BN + SiLU, NHWC bf16 out.  y->c in {16, 32, 48, 64, 96}. */
int yl_stem_conv(const float* x_nchw, int n, int ci, int h, int w, const void* w_packed, int ci_pad,
                 const float* bias, const yl_tensor* y, int act, void* stream);

/* DWConv (conv.py:100-105), depthwise 3x3 stride 1 pad 1 + folded BN (+SiLU): head.py:46-47, block.py:893.
 * w is bf16 [9][c]; optional residual-style `add` tensor is summed after activation (Attention: + pe(v)). */
int yl_dwconv3x3(const yl_tensor* x, const yl_tensor* y, const void* w, const float* bias, int act,
                 const yl_tensor* add, void* stream);

/* DWConv 3x3 + Conv 1x1 as one launch (csrc/dwpw_tc.cu): `nn.Sequential(DWConv(x, x, 3), Conv(x, c3, 1))` of the Detect class
 * branch (head.py:46-47), i.e. conv.py:100-105 followed by conv.py:47-49.  The depthwise conv (+ folded BN + SiLU) runs on
 * CUDA cores inside the producer of the 1x1 GEMM's A operand (depthwise result -> swizzled shared-memory tile -> tcgen05.mma),
 * so the intermediate tensor is never written.  `pw` describes the 1x1 conv whose `x` is the DEPTHWISE INPUT (same
 * dims as the depthwise output); dw_w is bf16 [9][x.c], dw_bias f32 [x.c] (yl_fold_bn_pack with depthwise = 1).
 * Needs x.c % 16 == 0, x.c <= 256, y.c <= 128, no residual / upsample / Detect epilogue. */
int yl_dw_pw_supported(const yl_conv_args* pw);
int yl_dw_pw_conv(const yl_conv_args* pw, const void* dw_w, const float* dw_bias, int dw_act, void* stream);
/* Back-to-back form for the LAST stage of the class branch on the engine path: DWConv 3x3 + Conv 1x1 + the head's final
 * nn.Conv2d(c3, nc, 1) (head.py:48) with its Detect epilogue, in one launch.  The 1x1 result (c3 channels) is not written:
 * the epilogue rounds it to bf16 into swizzled shared-memory tiles that are the A operand of a SECOND tcgen05 GEMM with the
 * head conv's weights, whose accumulator feeds the class decode / class filter.  `head`: the yl_conv_args of the final conv
 * with det.mode = YL_DET_CLS or YL_DET_CLS_FILTER and y.data == NULL (its x is ignored); head->x.c == pw->y.c <= 128,
 * nc <= 128.  Bit-identical to yl_dw_pw_conv followed by yl_conv_bn_act(head). */
int yl_dw_pw_det_supported(const yl_conv_args* pw, const yl_conv_args* head);
int yl_dw_pw_det(const yl_conv_args* pw, const void* dw_w, const float* dw_bias, int dw_act, const yl_conv_args* head, void* stream);

/* SPPF's three chained MaxPool2d(5,1,2) (block.py:182-184), -inf padding; y1=m(x), y2=m(y1), y3=m(y2). */
int yl_sppf_pool(const yl_tensor* x, const yl_tensor* y1, const yl_tensor* y2, const yl_tensor* y3, int k,
                 void* stream);

/* Attention core (block.py:905-914): qkv is (n,h,w,heads*(2*kd+hd)) with per-head channel groups [q|k|v];
 * out[(n,i), head*hd + c] = sum_j softmax_j(scale * q_i.k_j) v_j[c].  `+ pe(v)` and `proj` are separate calls. */
int yl_psa_attention(const yl_tensor* qkv, const yl_tensor* out, int heads, int key_dim, int head_dim,
                     float scale, void* stream);

/* ---- Detect decode --------------------------------------------------------------------------------------
 * Replaces Detect._inference + DFL + make_anchors + dist2bbox (head.py:95-126, block.py:51-69,
 * tal.py:326-350).  levels[i] is the raw head map of level i, NHWC f32 with 4*reg_max + nc channels
 * (box bins first).  y is dense fp32 (B, 4+nc, A), A = sum h_i*w_i, anchors ordered level-major,
 * row-major inside a level: y[:, :4] = (cx, cy, w, h) * stride, y[:, 4:] = sigmoid(cls). */
int yl_detect_decode(const yl_tensor* levels, int nl, const float* strides_host, int reg_max, int nc, float* y,
                     void* stream);
/* The same decode into a window of a wider prediction (the members of a model ensemble, Ensemble.forward nn/tasks.py,
 * concatenate their predictions along the anchor axis): y is dense fp32 (B, 4+nc, y_anchors) and the A = sum h_i*w_i
 * anchors land in columns [anchor_base, anchor_base + A); no other column is touched.  yl_detect_decode is this call
 * with (A, 0). */
int yl_detect_decode_into(const yl_tensor* levels, int nl, const float* strides_host, int reg_max, int nc, float* y,
                          int y_anchors, int anchor_base, void* stream);

/* Standalone DFL module (block.py:51-69): x dense fp32 (b, 4*reg_max, a) -> y (b, 4, a): softmax over the
 * reg_max bins of each side, expectation with weights 0..reg_max-1. */
int yl_dfl(const float* x, float* y, int b, int reg_max, int a, void* stream);

/* ---- NMS ------------------------------------------------------------------------------------------------
 * Replaces ops.non_max_suppression (utils/ops.py:138-273) including torchvision.ops.nms (ops.py:265):
 * candidate filter (strict >), best-class or multi-label expansion, optional class filter, max_nms top-k,
 * fp32 class offset `cls * max_wh`, stable descending sort, greedy IoU suppression with torchvision's CPU
 * arithmetic, first max_det survivors.  pred is dense fp32 (B, 4+nc, A), boxes as (cx, cy, w, h).
 * out: (B, max_det, 6) fp32 rows [x1,y1,x2,y2,conf,cls] in descending score order; counts: (B) int32.
 * classes_dev: optional int32[n_classes] device array (NULL = all classes). */
size_t yl_nms_workspace_bytes(int B, int A, int nc, int multi_label);
int yl_nms_batched(const float* pred, int B, int nc, int A, float conf_thres, double iou_thres,
                   const int32_t* classes_dev, int n_classes, int agnostic, int multi_label, int max_det,
                   int max_nms, float max_wh, void* workspace, size_t workspace_bytes, float* out,
                   int32_t* counts, void* stream);
/* yl_nms_batched with ground-truth priors, the `labels=` argument of ops.non_max_suppression (utils/ops.py:225-230,
 * passed by the validator's save_hybrid): label row l of image b, (cx, cy, w, h) in pred's pixel frame
 * label_xywh[label_offsets[b] + l] and class label_cls[...] in [0, nc) (not checked on the device), joins the
 * image's candidates after its anchors as a row with score 1.0 at its class: it survives when conf_thres < 1 and
 * the class filter admits it, and the max_nms cut, the class offsets and greedy NMS treat it like an anchor.
 * An image with no anchor above conf_thres still outputs its priors.  label_offsets (B+1) int32 device array;
 * max_labels_per_image bounds every image's count and sizes the workspace:
 * workspace >= yl_nms_priors_workspace_bytes(B, A, nc, multi_label, max_labels_per_image), and
 * (A + max_labels_per_image) * nc < 2^32.  label_offsets == NULL or max_labels_per_image == 0 is yl_nms_batched. */
size_t yl_nms_priors_workspace_bytes(int B, int A, int nc, int multi_label, int max_labels_per_image);
int yl_nms_batched_priors(const float* pred, int B, int nc, int A, float conf_thres, double iou_thres,
                          const int32_t* classes_dev, int n_classes, int agnostic, int multi_label, int max_det,
                          int max_nms, float max_wh, const float* label_xywh, const int32_t* label_cls,
                          const int32_t* label_offsets, int max_labels_per_image, void* workspace,
                          size_t workspace_bytes, float* out, int32_t* counts, void* stream);
/* torchvision.ops.nms semantics on explicit boxes (n,4) xyxy + scores (n): keep (int64[n]) gets the kept
 * indices in descending score order, *count their number.  workspace >= yl_nms_boxes_workspace_bytes(n). */
/* The two halves of yl_nms_batched for a step whose class filter runs inside the Detect head convs
 * (YL_DET_CLS_FILTER): yl_nms_begin zeroes the per-image candidate counters of `workspace` (before those convs),
 * yl_nms_select runs the per-image sort + greedy suppression on the candidates found there.  `pred` needs valid box
 * rows only.  Same outputs, bit for bit, as yl_nms_batched(multi_label = 0, classes = NULL) on the full tensor. */
int yl_nms_begin(void* workspace, size_t workspace_bytes, int B, void* stream);
/* Debug aid (tools/nms_phases.py): subsequent select launches of the calling thread accumulate, per image, the clock
 * cycles of their phases into device_buf[B][8] = {setup, round staging + sort, candidates vs kept, compaction, pairwise
 * mask, serial resolve, kept, candidates consumed}.  NULL disables.  Not for production use. */
int yl_debug_nms_phases(long long* device_buf);
int yl_nms_select(const float* pred, int B, int nc, int A, double iou_thres, int agnostic, int max_det, int max_nms,
                  float max_wh, void* workspace, size_t workspace_bytes, float* out, int32_t* counts, void* stream);
size_t yl_nms_boxes_workspace_bytes(int n);
int yl_nms_boxes(const float* boxes, const float* scores, int n, double iou_thres, void* workspace,
                 size_t workspace_bytes, int64_t* keep, int32_t* count, void* stream);
/* ops.py:213 in_place=True side effect: pred[:, :4] (cx,cy,w,h) -> (x1,y1,x2,y2), xywh2xyxy ops.py:372-389. */
int yl_xywh2xyxy_inplace(float* pred, int B, int C, int A, void* stream);
/* ops.scale_boxes + clip_boxes (utils/ops.py:66-98, 276-295) on the padded (B,max_det,6) detections:
 * per image: box -= (padx,pady); box /= gain; clamp to (0..w0, 0..h0).  params_dev: float[B][5] =
 * {gain, padx, pady, w0, h0}. */
int yl_scale_boxes(float* dets, const int32_t* counts, int B, int max_det, const float* params_dev, void* stream);

/* Elementwise widening of an image batch to fp32 (n elements): the `.float()` of engine/predictor.py:83 for fp16
 * (x_dtype == YL_F16: half the PCIe bytes of fp32) and, for x_dtype == YL_U8, `.float() / 255` (the `/255` of
 * predictor.py:84 / data/loaders.py:525-530; true fp32 division): a quarter of the PCIe bytes. */
int yl_to_f32(const void* x, int x_dtype, float* y, long long n, void* stream);

/* ---- fused stem --------------------------------------------------------------------------------------------- */
/* Image ingest + layer 0 + layer 1 (cfg/yolo11.yaml:17-18: Conv(3,c0,3,2) -> Conv(c0,c1,3,2), each conv+BN+SiLU,
 * nn/modules/conv.py:47-49) in one kernel: reads the caller's NCHW batch once, keeps the layer-0 map in
 * shared memory (bf16, same rounding as the unfused path) and writes only the layer-1 output y (n, h/4, w/4, c1).
 * x_dtype: YL_F32 (values used as they are), YL_F16 (widened), YL_U8 (image bytes: value / 255 in fp32, the
 * predictor's `/255`): the narrow types cut the ingest's HBM read (and the caller's PCIe upload) 2x / 4x.
 * w0 / w1: yl_fold_bn_pack outputs.  yl_stem_fused_supported(ci, c0, c1): built for ci <= 3, c0 = 16, c1 = 32. */
int yl_stem_fused_supported(int ci, int c0, int c1);
int yl_stem_fused(const void* x_nchw, int x_dtype, int n, int ci, int h, int w, const void* w0, int ci_pad0,
                  const float* b0, int act0, const void* w1, int ci_pad1, const float* b1, int act1, const yl_tensor* y,
                  void* stream);

/* ---- fused C3k2 tail ----------------------------------------------------------------------------------------- */
/* Everything after cv1 of a C3k2 / C2f block with ONE plain Bottleneck (nn/modules/block.py:231-235, 330-343,
 * 720-728): t = cv1(x) = [y0 | y1] (2c channels) ->
 *     h = SiLU(conv3x3_a(y1)) (c -> c/2);  y2 = [y1 +] SiLU(conv3x3_b(h)) (c/2 -> c);
 *     y = SiLU(conv1x1_2([y0, y1, y2])) (3c -> c2)
 * in one kernel: h and y2 never leave shared memory (bf16, the same rounding points as the layer-by-layer path).
 * wa / wb / w2 are yl_fold_bn_pack outputs ([co_pad][k*k*ci_pad] bf16) with their fp32 biases.
 * yl_c3k2_tail_supported(c, c2): built for c in {16, 32}, c2 in {32, 64, 128, 256}. */
int yl_c3k2_tail_supported(int c, int c2);
int yl_c3k2_tail(const yl_tensor* t, const yl_tensor* y, const void* wa, const float* ba, int wa_co_pad, int wa_ci_pad,
                 const void* wb, const float* bb, int wb_ci_pad, const void* w2, const float* b2, int w2_ci_pad,
                 int shortcut, void* stream);
/* The same block on tcgen05 (csrc/c3k2_tc.cu): intermediates stay in shared memory, each epilogue writes the swizzled
 * K-major tile that is the next tcgen05.mma's A operand.  Parity-tested; measured 1.5x slower than the mma.sync kernel on
 * these thin shapes (profiles/r02_c3k2_tc.md), so yl_c3k2_tail only dispatches to it under YL_C3K2_TC=1.  c in {16, 32},
 * c2 in {32, 64, 128}. */
int yl_c3k2_tail_tc(const yl_tensor* t, const yl_tensor* y, const void* wa, const float* ba, int wa_co_pad, int wa_ci_pad,
                 const void* wb, const float* bb, int wb_ci_pad, const void* w2, const float* b2, int w2_ci_pad,
                 int shortcut, void* stream);

/* ---- validator metric (the caller after the path, SURVEY §8f) ------------------------------------------------- */
/* box_iou (utils/metrics.py:51-70) + match_predictions (engine/validator.py:195-233, :410-429) for a whole batch:
 * dets (B,max_det,6) [x1,y1,x2,y2,conf,cls] + counts (B) as written by yl_nms_batched (already in label space),
 * gt_boxes (L,4) xyxy + gt_cls (L) fp32 for all images back to back, gt_offsets (B+1) int32 (image b owns labels
 * [gt_offsets[b], gt_offsets[b+1]), at most max_labels_per_image of them), iou_thresholds_dev (n <= 16, device).
 * tp (B,max_det,n) uint8: detection d is a true positive at threshold t.  Rows >= counts[b] are zero. */
int yl_match_predictions(const float* dets, const int32_t* counts, int B, int max_det, const float* gt_boxes,
                         const float* gt_cls, const int32_t* gt_offsets, int max_labels_per_image,
                         const float* iou_thresholds_dev, int n_thresholds, uint8_t* tp, void* stream);
/* ConfusionMatrix.process_batch (utils/metrics.py, called per image by the validator's update_metrics when
 * plots=True) for a whole batch, same dets / counts / labels layout as yl_match_predictions: the detections with
 * conf > `conf` are paired with labels of any class at box_iou > iou_thres; each detection keeps its highest-IoU
 * pair, then each label the highest-IoU pair left (exact ties: lower label index, then lower detection index).
 * Accumulates with integer atomics into matrix, int64[(nc+1)*(nc+1) + 1] on the device, indexed
 * [predicted * (nc+1) + true] with nc = background: matched label [cls(det), cls(gt)], unmatched label
 * [nc, cls(gt)], unmatched detection [cls(det), nc].  A class outside [0, nc] counts in the last element instead. */
int yl_confusion_matrix(const float* dets, const int32_t* counts, int B, int max_det, const float* gt_boxes,
                        const float* gt_cls, const int32_t* gt_offsets, int max_labels_per_image, int nc, float conf,
                        float iou_thres, int64_t* matrix, void* stream);

/* ---- image preprocess (the step before the path, SURVEY §8f) ---------------------------------------------- */
/* One source image of a letterbox batch: HWC uint8 BGR on the DEVICE, `pitch` bytes per row; it is resized to
 * (new_w, new_h) with cv2's 8-bit INTER_LINEAR arithmetic (skipped when the size already matches) and placed
 * at (left, top) of the output canvas. */
typedef struct yl_lb_image {
    const uint8_t* src;
    int32_t sh, sw, pitch;
    int32_t new_w, new_h, left, top;
    int32_t _pad;
} yl_lb_image;
/* LetterBox + BGR->RGB + HWC->CHW + float + /255 (data/augment.py:612-681, engine/predictor.py:67-85) for n
 * images into dst_nchw (n,3,H,W) fp32; canvas pixels outside an image get pad_value/255 (the reference pads
 * with 114).  Bit-exact against cv2.resize(INTER_LINEAR) + copyMakeBorder + the float conversion on the CPU.
 * imgs_dev: n descriptors in DEVICE memory. */
int yl_letterbox_u8(const yl_lb_image* imgs_dev, int n, float* dst_nchw, int H, int W, int pad_value, void* stream);

/* ---- test-time augmentation (DetectionModel._predict_augment, nn/tasks.py) -------------------------------------- */
/* One augmented input of _predict_augment: scale_img(x.flip(3) if flip else x, ratio, gs) (utils/torch_utils.py), i.e.
 * F.interpolate(bilinear, align_corners=False) to the content size (h, w) at the top-left of an (H, W) canvas whose other
 * pixels are F.pad's 0.447.  y: dense (n, c, H, W) fp32, 16-byte aligned, W % 4 == 0. */
typedef struct yl_tta_canvas {
    float* y;
    int32_t H, W;    /* canvas */
    int32_t h, w;    /* resized content (int(h * ratio), int(w * ratio)) */
    int32_t flip;    /* 1: left-right flip before the resize */
    int32_t _pad;
} yl_tta_canvas;
/* The scale_img calls of passes 1 and 2 of _predict_augment in ONE launch: x is the (n, c, h, w) batch in YL_F32,
 * YL_F16 (widened) or YL_U8 (value / 255 in fp32, the model input after the predictor's `/255`), read once for both
 * canvases[2].  Same arithmetic as ATen's upsample_bilinear2d; w <= 6144. */
int yl_tta_scale_img(const void* x, int x_dtype, int n, int c, int h, int w, const yl_tta_canvas* canvases, void* stream);
/* One pass of _predict_augment as seen by the merge: its prediction (B, 4+nc, A) fp32 and the anchors [a0, a0+n) that
 * _clip_augmented keeps. */
typedef struct yl_tta_pass {
    const float* pred;
    int32_t A;
    int32_t a0, n;
    int32_t flip;    /* 1: left-right flip (flips == 3 of _descale_pred) */
    float scale;     /* the pass's scale_img ratio */
    int32_t _pad;
} yl_tta_pass;
/* _descale_pred + _clip_augmented + torch.cat(y, -1) of _predict_augment over passes[3]: y (B, 4+nc, sum n) fp32 gets,
 * per pass in order, its kept anchors with rows 0..3 multiplied by the fp32 reciprocal of `scale` (torch's CUDA
 * `p[:, :4] /= scale`) and, for a flipped pass, row 0 replaced by img_w - x.  Bit-identical to those torch ops on CUDA. */
int yl_tta_merge(const yl_tta_pass* passes, int B, int nc, int img_w, float* y, void* stream);

/* ---- feature embeddings (BaseModel._predict_once with `embed`, nn/tasks.py) ------------------------------------ */
/* One tapped layer output: an NHWC bf16 channel slice (c, coff and cstride multiples of 8, data 16-byte aligned) whose
 * per-channel spatial mean fills output columns [col, col + c). */
typedef struct yl_embed_tap {
    yl_tensor x;
    int32_t col;
    int32_t _pad;
} yl_embed_tap;
/* adaptive_avg_pool2d(x, (1, 1)).squeeze(-1).squeeze(-1) of every tap, side by side in out (B, D) fp32, in ONE launch:
 * each element is the fp32 sum of the tap's h*w bf16 values times 1/(h*w).  taps: n_taps (<= 32) descriptors in HOST
 * memory, each with n == B.  Deterministic (no floating-point atomics; the pixel split is a function of h*w and c only).
 * workspace: NULL -> only writes the bytes it needs to *workspace_bytes (0 is possible) and returns.  Otherwise
 * *workspace_bytes is its capacity; it must be zeroed once before its first use, and every completed launch leaves it
 * zeroed again.  One workspace serves one launch at a time. */
int yl_embed_pool(const yl_embed_tap* taps, int n_taps, int B, int D, float* out, void* workspace, size_t* workspace_bytes,
                  void* stream);

/* ---- COCO bbox evaluation (the validator's save_json=True; pycocotools 2.0.x COCOeval, iouType="bbox") --------- */
/* The evaluated set in flat DEVICE arrays.  Pairs are the (category, image) pairs with at least one gt or dt, in
 * category-major order with image ranks (ascending image ids) ascending inside a category; gts and dts are CSR over
 * the pairs.  A pair's gts are in annotation-file order; its dts are its kept results: ordered by descending score with
 * ties in results-list order (np.argsort(-score, kind="mergesort")) and cut to maxDets[-1].  Every value is finite. */
typedef struct yl_cocoeval_set {
    int32_t n_pairs, n_cats, n_slots;  /* n_slots: kept dts in all */
    int32_t max_gt, max_dt;       /* largest gt group and largest kept dt group of one pair */
    const int32_t* pair_cat;      /* [n_pairs] category index */
    const int32_t* gt_off;        /* [n_pairs + 1] */
    const double* gt_bbox;        /* [n_gt][4] x, y, w, h */
    const double* gt_area;        /* [n_gt] the annotation's area (not w * h) */
    const uint8_t* gt_iscrowd;    /* [n_gt] */
    const int64_t* gt_id;         /* [n_gt] */
    const int32_t* slot_off;      /* [n_pairs + 1] CSR of the kept dts */
    const double* dt_bbox;        /* [n_slots][4] */
    const double* dt_score;       /* [n_slots] */
    const double* dt_area;        /* [n_slots] w * h (COCO.loadRes) */
    const int64_t* dt_id;         /* [n_slots] */
} yl_cocoeval_set;
/* COCOeval.params, DEVICE arrays: iouThrs[T], recThrs[R], areaRng[A][2] (A <= 16), maxDets[M] ascending. */
typedef struct yl_cocoeval_params {
    const double* iou_thrs;
    const double* rec_thrs;
    const double* area_rng;
    const int32_t* max_dets;
    int32_t T, R, A, M;
} yl_cocoeval_params;
/* Outputs of yl_cocoeval_evaluate per kept dt slot: an int64 key whose ascending order is descending score, its rank in
 * its pair, and flags[A][T][n_slots] with bit 0 = dtMatches != 0, bit 1 = dtIgnore; npig[K][A]: non-ignored gts per
 * category and area range. */
typedef struct yl_cocoeval_slots {
    int64_t* key;
    int32_t* rank;
    uint8_t* flags;
    int32_t* npig;
} yl_cocoeval_slots;
/* COCOeval.computeIoU + COCOeval.evaluateImg (maxDet = maxDets[-1]) of every pair in ONE launch: maskApi bbIou in
 * fp64, the greedy match with its quirks (equal IoU: the later gt in the ignore-sorted order wins; crowd gts match many
 * dts; a gt with id 0 leaves dtMatches = 0; area bounds inclusive).  Writes every kept slot and npig (zeroed first). */
int yl_cocoeval_evaluate(const yl_cocoeval_set* set, const yl_cocoeval_params* params, const yl_cocoeval_slots* out,
                         void* stream);
/* COCOeval.accumulate: one CTA per (category, area, maxDet, iouThr).  score[n_slots], rank[n_slots] and
 * flags[A][T][n_slots] hold the slots of evaluate in accumulate order: category by category (category k owns
 * [cat_slot_off[k], cat_slot_off[k+1])), each category's slots in np.argsort(-score, "mergesort") order over the
 * image-ascending concatenation.  Writes precision[T][R][K][A][M], recall[T][K][A][M] and scores[T][R][K][A][M] (fp64,
 * DEVICE), -1 where the category has no non-ignored gt; bit-identical to numpy. */
int yl_cocoeval_accumulate(const yl_cocoeval_params* params, int n_cats, int n_slots, const int32_t* cat_slot_off,
                           const double* score, const int32_t* rank, const uint8_t* flags, const int32_t* npig,
                           double* precision, double* recall, double* scores, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* YL11_H */
