/*
 * yolo_b200 -- C ABI of the B200-native YOLO decode + NMS hot path.
 *
 * The reference (Dipet/pytorch_yolo) is pure Python and has no FFI layer; its
 * boundary for this path is the Python API (YOLOLayer.forward,
 * non_max_suppression).  This header is the C ABI a binding for that API calls:
 * pytorch_yolo_b200/_lib.py binds it with ctypes, INTEGRATION.md shows the stub a
 * reference maintainer would add.  Each entry point cites the reference code it
 * replaces (paths relative to the reference root).
 *
 * Conventions
 *   - plain C: pointers and sizes only, no torch types; every pointer is a DEVICE
 *     pointer unless the name ends in _host;
 *   - the caller owns every buffer (inputs, outputs, workspace); the library never
 *     allocates, frees or synchronises; all work is enqueued on `stream`
 *     (a cudaStream_t; NULL = legacy default stream) and is CUDA-graph capturable;
 *   - return value: 0 = ok, < 0 = invalid argument (YOLO_B200_E_*), > 0 = cudaError_t
 *     of a failed launch;
 *   - re-entrant, no global state.
 */
#ifndef YOLO_B200_H
#define YOLO_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define YOLO_B200_ABI_VERSION 3
#define YOLO_B200_MAX_SCALES 4
#define YOLO_B200_MAX_ANCHORS 8      /* anchors per scale */
#define YOLO_B200_MAX_CLASSES 4096
#define YOLO_B200_DET_COLS 7         /* x1 y1 x2 y2 score cls_conf cls  (utils/utils.py:234) */

#define YOLO_B200_E_NULL      (-1)   /* null pointer */
#define YOLO_B200_E_RANGE     (-2)   /* size / count / threshold out of range */
#define YOLO_B200_E_ALIGN     (-3)   /* pointer not aligned as documented */
#define YOLO_B200_E_WORKSPACE (-4)   /* workspace too small */
#define YOLO_B200_E_UNSUPPORTED (-5) /* geometry outside what the fused head kernel covers: nothing was launched */

typedef struct CUstream_st* yolo_b200_stream_t;

/* One detection scale = one YOLOLayer (models/yolo_layer.py:25-111).
 * Constants are what YOLOLayer.create_grids computes (yolo_layer.py:101-111). */
typedef struct {
    const float* head;      /* (B, na*(5+nc), ny, nx) fp32 NCHW contiguous: the tensor YOLOLayer.forward receives.
                               yolo_b200_decode_compact_ex with YOLO_B200_VARIANT_F16 / _BF16 reads it as fp16 / bf16
                               elements instead (2-byte aligned; 8-byte aligned planes take 8-byte loads); with
                               YOLO_B200_VARIANT_NHWC it is (B, ny, nx, na*(5+nc)) contiguous (channels_last) */
    int32_t ny, nx;         /* grid size (p.shape[-2], p.shape[-1]) */
    int32_t na;             /* anchors of this layer (len(anchors)) */
    int32_t row_off;        /* first row of this scale inside one image of the concatenated prediction
                               (torch.cat(io, 1), models/yolov3_spp.py:163-164) */
    float stride;           /* img_size / max(nx, ny)           (yolo_layer.py:102) */
    float anchor_vec[YOLO_B200_MAX_ANCHORS][2];   /* anchors / stride, fp32 (yolo_layer.py:109) */
} yolo_b200_scale;

/* Per-candidate record, split in two 16-byte halves (32 bytes per candidate in total). */
typedef struct { float x1, y1, x2, y2; } yolo_b200_box;            /* xywh2xyxy output (utils.py:46-60) */
typedef struct {
    float score;            /* obj * max class conf            (utils.py:213) */
    float cls_conf;         /* max class conf                  (utils.py:212) */
    int32_t cls;            /* first arg-max class             (utils.py:212) */
    int32_t row;            /* anchor row inside the image (0 .. N-1) -- the tie-break key */
} yolo_b200_meta;

int yolo_b200_abi_version(void);
const char* yolo_b200_error_string(int code);

/* Dense decode: replaces YOLOLayer.forward's eval branch for every scale plus the model-level
 * torch.cat (yolo_layer.py:90-99, yolov3_spp.py:163-164).
 * io: (B, rows_per_img, 5+nc) fp32, written once.  Reads each head element once.
 * n_classes <= 434 (one 128-position tile of 5+nc channel rows is staged in shared memory). */
int yolo_b200_decode_dense(const yolo_b200_scale* scales_host, int n_scales, int batch, int n_classes,
                           int rows_per_img, float* io, yolo_b200_stream_t stream);
/* Same call with an explicit kernel variant: 0 = automatic, 1 = LDG kernel (one CTA per 128-position tile, load phase then
 * store phase), 2 = TMA kernel (persistent CTAs: tensor-map tile loads into a shared-memory ring, transposed tiles leave
 * as bulk copies shared -> global; needs 5+n_classes <= 150).  Identical results.  Automatic picks the TMA kernel for
 * the scales whose planes are a multiple of 4 floats when 5+n_classes <= 150, the LDG kernel for everything else.  A call
 * refused with an argument error (YOLO_B200_E_*) enqueues nothing: io keeps what it held. */
int yolo_b200_decode_dense_ex(const yolo_b200_scale* scales_host, int n_scales, int batch, int n_classes,
                              int rows_per_img, float* io, int variant, yolo_b200_stream_t stream);

/* Fused decode + confidence filter + stream compaction: YOLOLayer.forward (eval) + cat +
 * the first half of non_max_suppression (utils.py:210-234) without materialising the
 * (B, N, 5+nc) tensor.  Candidates of image b land in slots [b*cap, b*cap + min(count[b], cap));
 * count[b] is the number that passed (may exceed cap: then *overflow != 0 and the excess is dropped).
 * count (batch ints) and overflow (1 int) are zeroed by the call itself. */
int yolo_b200_decode_compact(const yolo_b200_scale* scales_host, int n_scales, int batch, int n_classes,
                             int rows_per_img, float conf_thres, float min_wh,
                             yolo_b200_box* cand_box, yolo_b200_meta* cand_meta, int cap_per_img,
                             int32_t* count, int32_t* overflow, yolo_b200_stream_t stream);

/* Same call with an explicit kernel variant: 0 = automatic (= 1), 1 = gated LDG kernel (many small CTAs, 128-bit
 * coalesced loads; reads the objectness plane first and the box and class planes only around positions whose objectness
 * can pass conf_thres), 2 = TMA kernel (persistent CTAs, ring of 1-D cp.async.bulk copies; needs 5+n_classes <= 800),
 * 3 = the same kernel fed by one 2-D tensor-map copy per tile (needs 5+n_classes <= 256), 4 = dense LDG kernel (variant 1
 * without the gate: reads every plane).  Variants 2 to 4 read the whole head tensor.  All produce identical candidates.
 * A call refused with an argument error (YOLO_B200_E_*) enqueues nothing: count and overflow keep what they held. */
int yolo_b200_decode_compact_ex(const yolo_b200_scale* scales_host, int n_scales, int batch, int n_classes,
                                int rows_per_img, float conf_thres, float min_wh,
                                yolo_b200_box* cand_box, yolo_b200_meta* cand_meta, int cap_per_img,
                                int32_t* count, int32_t* overflow, int variant, yolo_b200_stream_t stream);

/* OR-ed into `variant`: do not zero count / overflow first -- the candidates are appended to what earlier calls on the
 * same buffers produced (used when some scales of a model go through yolo_b200_head_decode_compact). */
#define YOLO_B200_VARIANT_ACCUMULATE 0x100
/* OR-ed into `variant` of yolo_b200_decode_compact_ex: every scale.head of the call holds fp16 (F16) or bf16 (BF16) elements.
 * Each value is converted to fp32 as it is loaded, exactly, so the candidates are bit-identical to those of the same call on
 * the fp32 upcast of the heads (this decodes in fp32; the reference run on 16-bit tensors rounds every op to 16 bits).
 * Variants 0, 1 and 4 take them; with variant 2 or 3 the call returns YOLO_B200_E_UNSUPPORTED, with both bits
 * YOLO_B200_E_RANGE, before anything is enqueued.  The other entry points read fp32 only. */
#define YOLO_B200_VARIANT_F16 0x200
#define YOLO_B200_VARIANT_BF16 0x400
/* OR-ed into `variant` of yolo_b200_decode_compact_ex: every scale.head of the call holds the channels_last (NHWC) memory of
 * its (B, na*(5+nc), ny, nx) tensor, i.e. (B, ny, nx, na*(5+nc)) contiguous -- what a torch.channels_last model hands over.
 * It is read in place by a kernel that streams those rows of 5+nc logits through a shared-memory ring (one bulk copy per
 * tile; a head whose base is not 16-byte aligned takes plain loads) and reads every byte.  The candidates are bit-identical
 * to those of the same call on the NCHW copy of the heads.  Combines with variant 0, _ACCUMULATE, _F16 and _BF16; with
 * variants 1 to 4 (NCHW kernels) the call returns YOLO_B200_E_UNSUPPORTED before anything is enqueued. */
#define YOLO_B200_VARIANT_NHWC 0x1000

/* Same candidates, from an already decoded prediction (the tensor model.forward returned):
 * utils.py:210-234.  With write_back_score != 0 the product obj*max_cls is stored into
 * pred[..., 4] exactly like the reference's in-place update (utils.py:213). */
int yolo_b200_compact_from_dense(float* pred, int batch, int rows_per_img, int n_classes,
                                 float conf_thres, float min_wh, int write_back_score,
                                 yolo_b200_box* cand_box, yolo_b200_meta* cand_meta, int cap_per_img,
                                 int32_t* count, int32_t* overflow, yolo_b200_stream_t stream);

/* Segmented NMS: per image, per class: order by (score desc, row asc), keep the first
 * max_per_class (100, utils.py:247-250), greedy suppression with strict IoU > nms_thres and the
 * score-weighted 'MERGE' box (utils.py:266-275, bbox_iou utils.py:63-96), then the per-image
 * ordering by score (utils.py:289-291; ties: class asc, then in-class order).
 * out:       (batch, out_cap, 7) fp32 rows, image b holds out_count[b] rows
 * out_row:   (batch, out_cap) anchor row of each kept detection
 * out_count: (batch) number of detections (0 <=> the reference returns None for that image)
 * out_cap must be >= min(cap_per_img, n_classes * max_per_class).
 * out / out_row / out_count may live in a peer GPU's memory (NVLink peer stores). */
size_t yolo_b200_nms_workspace_bytes(int batch, int cap_per_img, int n_classes, int max_per_class);
int yolo_b200_nms(const yolo_b200_box* cand_box, const yolo_b200_meta* cand_meta, const int32_t* count,
                  int batch, int cap_per_img, int n_classes, float nms_thres, int max_per_class,
                  float* out, int32_t* out_row, int out_cap, int32_t* out_count,
                  void* workspace, size_t workspace_bytes, yolo_b200_stream_t stream);

/* Same call with options.  step_seq / step_stamp (both or neither): a completion stamp for the multi-GPU gather -- once
 * every result row of the call has been stored, the kernel writes ++*step_seq to *step_stamp with release semantics at
 * system scope.  step_seq is a zero-initialised int32 in this GPU's memory that belongs to the (lane, caller) pair;
 * step_stamp may live in a peer GPU's memory next to out / out_row / out_count, where yolo_b200_flag_wait polls it. */
typedef struct {
    int32_t flags;          /* reserved, 0 */
    int32_t seg_warps_per_sm; /* resident single-warp CTAs per SM of the segment kernel, 1..32; 0 = default (16) */
    int32_t* step_seq;
    int32_t* step_stamp;
} yolo_b200_nms_opts;
int yolo_b200_nms_ex(const yolo_b200_box* cand_box, const yolo_b200_meta* cand_meta, const int32_t* count,
                     int batch, int cap_per_img, int n_classes, float nms_thres, int max_per_class,
                     float* out, int32_t* out_row, int out_cap, int32_t* out_count,
                     void* workspace, size_t workspace_bytes, const yolo_b200_nms_opts* opts /* may be NULL */,
                     yolo_b200_stream_t stream);

/* ---- head 1x1 convolution fused with decode + compaction (SURVEY.md section 8f, third "next" row) --------------
 * The producer of a head tensor is a 1x1 convolution over the last feature map: ConvBlock = conv (no bias) + BatchNorm +
 * LeakyReLU(0.1) in models/yolov3_spp.py:86,99,111 (models/yolo_base.py:19-44), a plain nn.Conv2d with bias in
 * models/yolov3_tiny.py:38,42.  This entry point computes it on the tcgen05 tensor cores (TF32 inputs, fp32 accumulate --
 * the precision cuDNN uses for the reference's convolution under torch's default allow_tf32) and decodes straight from
 * the accumulator: the (B, na*(5+nc), ny, nx) head tensor never reaches HBM unless head_out asks for it.
 * The caller folds an eval-mode BatchNorm into weight/bias (what ConvBlock.fuse does, models/yolo_base.py:46-57). */
typedef struct {
    const float* x;          /* (B, c_in, ny, nx) fp32 NCHW contiguous, 16-byte aligned: input of the head convolution.
                                With YOLO_B200_HEAD_F16 / _BF16: fp16 / bf16 elements, (B, c_in, pitch).  With
                                YOLO_B200_HEAD_NHWC: (B, ny, nx, c_in) contiguous (channels_last) */
    const float* weight;     /* (256, c_in) fp32 row-major, 16-byte aligned: rows na*(5+nc) .. 255 zero (the kernel's W tile
                                covers up to 256 output channels; which rows it fetches depends on the instantiation);
                                (512, c_in) with YOLO_B200_HEAD_FP32X3; (256, c_in) of x's 16-bit type with YOLO_B200_HEAD_F16 /
                                _BF16 */
    const float* bias_host;  /* HOST pointer: na*(5+nc) floats */
    float* head_out;         /* optional: (B, na*(5+nc), ny, nx) activated head tensor (what YOLOLayer.forward receives), or NULL */
    int32_t c_in;            /* multiple of 32 (16-bit x: of 64) */
    int32_t x_row_pitch;     /* elements between consecutive channel planes of x; 0 = ny*nx (contiguous NCHW).  16-bit x: when
                                given, a multiple of 8 (a 16-byte row pitch); contiguous planes that are not a multiple of 8
                                elements are read in place when even (38x38, 26x26, 19x20 ...), odd ones (19x19, 13x13) need
                                the padded copy of yolo_b200_pad_planes_16.  fp32 x: when given it must be
                                a multiple of 4 (TMA row pitch of 16 bytes).  A contiguous 19x19 or 13x13 map (361 / 169 floats
                                per plane) has no such pitch: the one-pass single-CTA kernel reads it in place with loader warps
                                (4-byte asynchronous copies); the three-pass mode and the CTA-pair kernel take it as a
                                (B, c_in, pitch) copy padded to 364 / 172 floats per plane (yolo_b200_pad_planes) */
    float negative_slope;    /* LeakyReLU slope in [0, 1]: 0.1 for ConvBlock heads, 1 for a plain convolution */
    yolo_b200_scale scale;   /* grid, anchors, stride, row_off of this YOLOLayer; scale.head is ignored */
} yolo_b200_head;

#define YOLO_B200_HEAD_ACCUMULATE    1   /* flags: append to count / overflow instead of zeroing them first */
#define YOLO_B200_HEAD_NO_CANDIDATES 2   /* flags: convolution only (head_out), no decode / compaction */
#define YOLO_B200_HEAD_CTA_PAIR       4   /* flags: use the tcgen05 cta_group::2 kernel (two CTAs share a 256-position tile and
                                            each stages half of the weights) where it is instantiated (3 anchors x 80 classes);
                                            same results, measured ~5 % slower than the default single-CTA kernel on B200 */
#define YOLO_B200_HEAD_FP32X3          8   /* flags: fp32-accurate products from three TF32 passes (operand split): every head's
                                            `weight` then holds 512 rows -- rows 256 .. 511 = w - trunc_tf32(w) of rows 0 .. 255,
                                            trunc_tf32 = clear the low 13 mantissa bits -- and the head tensor matches an fp32
                                            convolution to accumulation accuracy (about three times the tensor time) */
/* flags: x and weight hold fp16 (F16) or bf16 (BF16) elements.  The products run on tcgen05.mma kind::f16 (exact products of
 * the 16-bit operands, fp32 accumulation); bias, activation, decode and head_out stay fp32, and the candidates are
 * bit-identical to yolo_b200_decode_compact on the head tensor the same call writes to head_out.  One-pass single-CTA
 * kernel only; every return code is decided before anything is enqueued (count and overflow keep what they held):
 *   both bits: YOLO_B200_E_RANGE;  either bit with YOLO_B200_HEAD_FP32X3 or _CTA_PAIR: YOLO_B200_E_UNSUPPORTED;
 *   c_in % 64 != 0, an odd contiguous plane, or an x_row_pitch that is not a multiple of 8: YOLO_B200_E_UNSUPPORTED;
 *   x or weight not 16-byte aligned: YOLO_B200_E_ALIGN. */
#define YOLO_B200_HEAD_F16           0x10
#define YOLO_B200_HEAD_BF16          0x20
/* flags: every x is a channels_last (NHWC) feature map, (B, ny, nx, c_in) contiguous -- what a torch.channels_last model hands
 * over.  x is then a row-major (B*ny*nx, c_in) matrix: one 3-D tensor-map box per k-block brings 128 positions x 128 bytes of
 * channels (K-major, SWIZZLE_128B; the ragged last tile of an image is zero-filled), so every plane size (19x19, 13x13, odd
 * 16-bit planes) is read in place with no loader warps and no padded copy.  Same head values and candidates as the NCHW call.
 * Combines with YOLO_B200_HEAD_FP32X3, _F16 and _BF16; c_in, anchor and class rules as without it.  Every return code is
 * decided before anything is enqueued:  x_row_pitch != 0 or _CTA_PAIR: YOLO_B200_E_UNSUPPORTED;  x not 16-byte aligned:
 * YOLO_B200_E_ALIGN. */
#define YOLO_B200_HEAD_NHWC          0x40
#define YOLO_B200_HEAD_PROFILE_MAINLOOP 0x100  /* flags, profiling only (results are garbage): skip the epilogue */
#define YOLO_B200_HEAD_PROFILE_NO_W     0x200  /* profiling only: the weight tiles are fetched once, not per position tile */
#define YOLO_B200_HEAD_PROFILE_NO_X     0x400  /* profiling only: the feature tiles are fetched once */
#define YOLO_B200_HEAD_PROFILE_NO_MMA   0x800  /* profiling only: no tensor-core work, the stages are only recycled (stream rate) */

/* (rows, plane) floats -> (rows, pitch) floats, pitch >= plane and pitch % 4 == 0, pad columns zero: gives a feature map
 * whose planes are not a multiple of 4 floats (19x19, 13x13) the 16-byte row pitch the fused head kernel's TMA loads need.
 * x 4-byte aligned, out 16-byte aligned. */
int yolo_b200_pad_planes(const float* x, float* out, long long rows, int plane, int pitch, yolo_b200_stream_t stream);
/* The same for 2-byte elements (fp16 / bf16 feature maps): (rows, plane) -> (rows, pitch), pitch >= plane and pitch % 8 == 0,
 * pad columns zero.  x 2-byte aligned, out 16-byte aligned. */
int yolo_b200_pad_planes_16(const void* x, void* out, long long rows, int plane, int pitch, yolo_b200_stream_t stream);

/* 1 when the fused kernel covers this geometry: c_in % 32 == 0, a row pitch x_row_pitch % 4 == 0 or contiguous planes, and
 * 3 anchors with 3*(5+n_classes) <= 256 (80, 20 and 1 classes have fully unrolled epilogues, any other count up to 80
 * runs a kernel with a run-time class loop).  Other scales go through the caller's own convolution +
 * yolo_b200_decode_compact_ex(... | YOLO_B200_VARIANT_ACCUMULATE). */
int yolo_b200_head_supported(int c_in, int ny, int nx, int x_row_pitch, int na, int n_classes);
/* the same question for a call with `flags` (YOLO_B200_HEAD_FP32X3, YOLO_B200_HEAD_CTA_PAIR: those need a 16-byte row pitch;
 * YOLO_B200_HEAD_F16 / _BF16: c_in % 64 == 0 and an 8-element pitch or even contiguous planes, see yolo_b200_head.x_row_pitch;
 * 0 for both 16-bit bits or for a 16-bit bit with FP32X3 or CTA_PAIR; YOLO_B200_HEAD_NHWC: every plane size, x_row_pitch == 0,
 * not with CTA_PAIR) */
int yolo_b200_head_supported_ex(int c_in, int ny, int nx, int x_row_pitch, int na, int n_classes, int flags);
/* Candidates exactly as yolo_b200_decode_compact would produce from the head tensor (same record layout, same count /
 * overflow protocol).  Every wait inside the kernel's pipeline is bounded (10 s of wall-clock time without progress):
 * a pipeline bug traps -- the launch fails and the next synchronisation on the stream reports the error -- instead of
 * hanging the GPU.  All heads with the same anchor count share
 * one persistent launch (tiles of every scale, heaviest first). */
int yolo_b200_head_decode_compact(const yolo_b200_head* heads_host, int n_heads, int batch, int n_classes, int rows_per_img,
                                  float conf_thres, float min_wh,
                                  yolo_b200_box* cand_box, yolo_b200_meta* cand_meta, int cap_per_img,
                                  int32_t* count, int32_t* overflow, int flags, yolo_b200_stream_t stream);

/* ---- post-NMS epilogue (SURVEY.md section 8f, first "next" row) ---------------------------------------------
 * scale_coords (utils/utils.py:296-303) + the .round() of _dict_from_results (utils.py:313), in place:
 *   x -= pad_x, y -= pad_y, /= gain, clamp(min=0), optional round-half-even; pad and gain are the fp32 values of
 *   the reference's python scalars: gain = max(img1)/max(img0), pad = (img1 - img0*gain)/2.
 * yolo_b200_scale_coords: one (n,4) box view whose rows are row_stride floats apart (7 for a detection tensor).
 * yolo_b200_scale_detections: every image of a yolo_b200_nms result in one launch; params = batch x (pad_x, pad_y,
 * gain) fp32 on the device. */
int yolo_b200_scale_coords(float* coords, int n, int row_stride, float pad_x, float pad_y, float gain,
                           int do_round, yolo_b200_stream_t stream);
int yolo_b200_scale_detections(float* out, const int32_t* out_count, int batch, int out_cap,
                               const float* params, int do_round, yolo_b200_stream_t stream);

/* ---- training-side consumer of the YOLOLayer constants (SURVEY.md section 8f, fourth "next" row) ---------------------
 * build_targets (utils/utils.py:160-197 with wh_iou, utils.py:99-121) for every YOLO layer of a model in one launch:
 * per layer the best anchor of each target by width/height IoU against anchor_vec, the iou_thres filter (target order
 * preserved) and the index / regression targets compute_loss reads.  targets: (nt, 6) fp32 [image, class, x, y, w, h]
 * (x, y, w, h relative to the image).  Per layer the caller provides room for nt entries; count[l] receives how many
 * survived.  Index outputs are int64 (torch.long), like the reference's. */
typedef struct {
    int32_t nx, ny;         /* layer.n_grids = (nx, ny)                       (yolo_layer.py:110) */
    int32_t na;             /* anchors of the layer */
    int32_t reserved;
    float anchor_vec[YOLO_B200_MAX_ANCHORS][2];   /* layer.anchor_vec        (yolo_layer.py:109) */
    int64_t *b, *a, *gj, *gi;   /* indices[l] = (image, anchor, grid y, grid x), nt entries each   (utils.py:185) */
    int64_t* tcls;              /* (nt)                                                           (utils.py:194) */
    float* txy;                 /* (nt, 2) gxy - floor(gxy)                                        (utils.py:188) */
    float* twh;                 /* (nt, 2) log(gwh / anchor_vec[a])                                (utils.py:191) */
} yolo_b200_target_layer;
int yolo_b200_build_targets(const float* targets, int nt, const yolo_b200_target_layer* layers_host, int n_layers,
                            float iou_thres, int32_t* count /* n_layers ints */, yolo_b200_stream_t stream);

/* ---- multi-GPU set-up (one process per GPU; not on the per-batch path) --------------------------
 * The reference has no multi-GPU code (SURVEY.md section 2.3).  Images are independent: every rank
 * runs the calls above on its slice, passing as out/out_row/out_count pointers into the ROOT rank's
 * result buffer, mapped here through CUDA IPC, so kept rows cross NVLink as peer stores issued by
 * the finalize kernel -- the "ragged gather" -- and no collective runs on the hot path.
 * These are the only entry points that allocate or map memory. */
#define YOLO_B200_PEER_HANDLE_BYTES 64
int yolo_b200_device_alloc(size_t bytes, void** out_dev_ptr);             /* cudaMalloc'd, exportable */
int yolo_b200_device_free(void* dev_ptr);
int yolo_b200_peer_export(void* dev_ptr, void* handle_out_host /*64 B*/); /* root: handle to broadcast */
int yolo_b200_peer_open(const void* handle_host /*64 B*/, void** out_mapped_ptr);  /* non-root ranks */
int yolo_b200_peer_close(void* mapped_ptr);


/* Step flags of the gather (per-batch path, no host involvement, CUDA-graph replayable): int32 sequence numbers in device
 * memory, possibly a peer's.  Every call site owns a zero-initialised device counter `seq` that the kernel itself
 * advances, so the enqueued work is identical from step to step.
 *   yolo_b200_flag_wait: ++*seq, then wait until flags[i] >= *seq + bias for all i < n_flags (acquire, system scope).
 *                        After timeout_s seconds the kernel gives up and stores 1 + (index of the missing flag) to *err.
 *   yolo_b200_flag_post: ++*seq, then *flag = *seq + bias (release, system scope): everything enqueued on `stream`
 *                        before the call is visible to whoever acquires the flag. */
int yolo_b200_flag_wait(const int32_t* flags, int n_flags, int32_t* seq, int bias, int32_t* err /* may be NULL */,
                        double timeout_s, yolo_b200_stream_t stream);
int yolo_b200_flag_post(int32_t* flag, int32_t* seq, int bias, yolo_b200_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* YOLO_B200_H */
