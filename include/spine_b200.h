/*
 * spine_b200.h -- C ABI of libspine_b200.so: the sm_100a implementation of
 * spine-vision's localization-and-crop hot path.
 *
 * The reference (nghiant03/spine-vision, pure Python) has no FFI layer; the
 * path sits behind plain Python callables.  Each entry point below replaces
 * the device-side work of the reference callables it cites (paths relative to
 * the reference root).  The Python host mirror in spine_vision_b200/ binds
 * these with ctypes (see INTEGRATION.md for the stub a maintainer would add).
 *
 * Conventions
 *  - every pointer named d_* is a DEVICE pointer owned by the caller
 *    (PyTorch tensors: tensor.data_ptr()); workspaces are caller-owned too.
 *    The library owns only svb_model and svb_model_graph handles.
 *  - calls are asynchronous on `stream` (a cudaStream_t passed as void*),
 *    with no hidden synchronisation or allocation, except svb_model_create /
 *    svb_model_destroy which allocate and synchronise, and
 *    svb_model_graph_create which allocates.
 *  - return value: 0 on success, negative svb_status otherwise; the message
 *    is available from svb_last_error() (thread local).  Nothing throws.
 *  - there is no CPU fallback: a device that is not sm_100 gives
 *    SVB_ERR_UNSUPPORTED_DEVICE.
 *  - a handle is bound to the device current at creation and is not
 *    thread-safe; one process per GPU.
 */
#ifndef SPINE_B200_H_
#define SPINE_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SVB_VERSION 100 /* 0.1.0 */

typedef enum svb_status {
    SVB_OK = 0,
    SVB_ERR_INVALID_ARG = -1,
    SVB_ERR_CUDA = -2,
    SVB_ERR_UNSUPPORTED_DEVICE = -3,
    SVB_ERR_WORKSPACE_TOO_SMALL = -4,
    SVB_ERR_BOX_TOO_LARGE = -5,
    SVB_ERR_MISSING_WEIGHT = -6,
    SVB_ERR_UNSUPPORTED_MODEL = -7,
    SVB_ERR_IO = -8,    /* host input / output stage: file cannot be opened, read or written */
    SVB_ERR_FORMAT = -9 /* host input stage: not a (supported) MetaImage file */
} svb_status;

typedef enum svb_dtype {
    SVB_BF16 = 0, /* bf16 operands, fp32 accumulate (BASELINE.json north_star) */
    SVB_FP16 = 1, /* fp16 operands, fp32 accumulate: same tensor rate, 3 more mantissa bits */
    SVB_F32 = 2   /* float32 -- output type of svb_k4_classifier_input only */
} svb_dtype;

int svb_version(void);
const char* svb_last_error(void);
/* 0 if the current CUDA device is sm_100 (B200), else SVB_ERR_UNSUPPORTED_DEVICE. */
int svb_device_check(void);
/* Number of CUDA kernels this library has launched in the process (all streams); reset != 0 zeroes the
 * counter after reading.  Instrumentation only (bench.py reports it as gpu_launches). */
long long svb_launch_count(int reset);

/* ------------------------------------------------------------------------------------------
 * K0 -- middle sagittal plane of the 0.3 mm isotropic resample, computed from the source volume.
 * Replaces resample_to_isotropic + extract_middle_slice + get_slice_spacing
 * (spine_vision/datasets/classification/cropping.py:37-101: SimpleITK ResampleImageFilter with an identity
 * transform and sitkLinear over the WHOLE volume, DICOMOrient(LPI), arr[:, :, n // 2]) for the one plane that is kept.
 * Parity is UNPINNED: SimpleITK is absent from the build image; the arithmetic is the restatement in
 * oracle/itk_resample.py (continuous index (i * new_spacing) / spacing, inside test [-0.5, size - 0.5), clamped
 * neighbours, nested double lerp x -> y -> z, default pixel 0, cast to float32).
 * The host resolves orientation and the fixed (Left-Right) axis (spine_vision_b200.volumes.plan_midplane).
 *
 *  d_volumes : float32 pool; series b is the array [nz][ny][nx] (sitk.GetArrayFromImage order) at vol_off
 *  d_desc    : svb_k0_series [B] on the device
 *  d_out     : float32 pool of output planes [out_h][out_w] at out_off -- the SlicePool K1 and K3 take
 */
typedef struct svb_k0_series {
    int64_t vol_off, out_off;          /* element offsets into d_volumes / d_out */
    int32_t nx, ny, nz;                /* size of the (possibly slab-cut) source array */
    int32_t ax_row, ax_col, ax_fix;    /* image axis (0 = x, 1 = y, 2 = z) running down the rows / across the columns / fixed */
    int32_t flip_row, flip_col;        /* the oriented axis runs against the image axis */
    int32_t out_h, out_w;              /* resampled sizes of the row / column axes: int(round(size * spacing / 0.3)) */
    int32_t fix_lo, fix_hi, fix_inside;       /* the two source planes around the fixed index (indices into the array) */
    int32_t integer_pixels;            /* the source pixel type is integral: ITK casts the interpolated double back to it
                                          (static_cast, i.e. truncation toward zero) -- the plane then holds whole numbers */
    double fix_frac;                   /* interpolation fraction between them */
    double sp_row, sp_col;             /* source spacing (mm) of the row / column axes */
    double new_sp_row, new_sp_col;     /* target spacing (0.3 mm) */
} svb_k0_series;
size_t svb_k0_workspace_bytes(int B, int max_out_h, int max_out_w);
int svb_k0_midplane_resample(const float* d_volumes, const svb_k0_series* d_desc, int B, int max_out_h,
                             int max_out_w, float* d_out, void* d_ws, size_t ws_bytes, void* stream);

/* K0 + K1 in one call (SURVEY 8f row 1: "fuse into K1"): source planes -> isotropic middle planes (kept: K3 cuts its crops from
 * them) + the uint8 model planes.  Replaces resample_to_isotropic + extract_middle_slice (cropping.py:37-79) AND
 * normalize_to_uint8 + Resize of predict_ivd_locations (io/__init__.py:15-30, cropping.py:463-472) for a batch.  K0 accumulates
 * every plane's min / max while it writes it, so K1 makes no min/max pass (SVB_K1_GROUP=n walks the batch in groups of n
 * planes that the resize launch reads back from L2: less DRAM traffic, more and smaller launches -- measured slower, off by
 * default).  d_offs / d_hw describe the planes in d_slices (= desc.out_off, out_h, out_w). */
size_t svb_k01_workspace_bytes(int B, int max_out_h, int max_out_w, int out_h, int out_w);
int svb_k01_midplane_normalize_resize(const float* d_volumes, const svb_k0_series* d_desc, int B, int max_out_h,
                                      int max_out_w, float* d_slices, const int64_t* d_offs, const int32_t* d_hw,
                                      int out_h, int out_w, uint8_t* d_out_u8, float* d_minmax, void* d_ws,
                                      size_t ws_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * K1 -- fused min-max normalise + antialiased bilinear resize to uint8.
 * Replaces, per slice: normalize_to_uint8 (spine_vision/io/__init__.py:15-30) followed by
 * PIL "L"->"RGB" + torchvision Resize (Pillow BILINEAR with antialias, uint8 fixed point)
 * in predict_ivd_locations (spine_vision/datasets/classification/cropping.py:463-472).
 * The three RGB planes are identical, so one plane is produced; /255 and mean/std are
 * folded into the model's stem (svb_model_create).
 *
 *  d_slices : float32 pool holding every slice, slice b starts at element d_offs[b]
 *  d_offs   : int64 [B]   element offsets into d_slices
 *  d_hw     : int32 [B,2] (height, width) of each slice
 *  max_h/w  : host-side maxima over the batch (launch sizing only)
 *  d_out_u8 : uint8 [B, out_h, out_w]
 *  d_minmax : float32 [B,2] (min, max) of each slice -- written, may be NULL
 *  d_ws     : workspace of at least svb_k1_workspace_bytes(...) bytes
 */
size_t svb_k1_workspace_bytes(int B, int max_h, int max_w, int out_h, int out_w);
int svb_k1_normalize_resize(const float* d_slices, const int64_t* d_offs, const int32_t* d_hw, int B,
                            int max_h, int max_w, int out_h, int out_w, uint8_t* d_out_u8,
                            float* d_minmax, void* d_ws, size_t ws_bytes, void* stream);

/* Normalise only (no resize): normalize_to_uint8 (io/__init__.py:15-30) over a ragged batch, as the localization dataset
 * builder applies it to every RSNA DICOM slice and Lumbar-Coords array before saving a PNG
 * (spine_vision/datasets/localization.py:147-151, 262-267).  d_out_u8 is a uint8 pool with the SAME element offsets as
 * the float32 pool (d_offs); bit-exact like K1's first half.  HBM-bound: 4 B in (twice: min/max, then normalise) + 1 B out. */
size_t svb_normalize_u8_workspace_bytes(int B);
int svb_normalize_u8(const float* d_slices, const int64_t* d_offs, const int32_t* d_hw, int B, int max_h, int max_w,
                     uint8_t* d_out_u8, float* d_minmax, void* d_ws, size_t ws_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * K3 -- batched coordinate-driven crop + per-crop min-max normalise + letterboxed bilinear
 * resize (OpenCV 8U INTER_LINEAR fixed point), plus the classifier's Pillow bilinear
 * Resize of the crop as an optional second output.
 * Replaces CropContext.crop -> crop_region_horizontal (cropping.py:316-354, 377-404) with
 * normalize_to_uint8 (io/__init__.py:15-30) and resize_with_padding (cropping.py:104-146),
 * and the Resize step of ClassificationDataset._build_transforms
 * (spine_vision/training/datasets/classification.py:247-278) for one channel.
 *
 *  d_slice_idx : int32 [N]   which slice each crop is cut from
 *  d_xy        : float32 [N,2] normalised (x, y) centre in [0,1] (model output; widened to double like the reference's
 *                float(output_np[i, 0]), cropping.py:481-483) -- or float64 [N,2] with SVB_K3_XY_F64, for centres that are
 *                Python floats in the reference (get_center_fallback_locations, cropping.py:486-492): int(x * w) must
 *                see the same double
 *  d_delta_px  : int32 [N,4] (left, right, top, bottom) from mm_to_pixels (cropping.py:149-169)
 *  d_crops     : uint8 [N, ch, cw]
 *  d_crops2    : uint8 [N, oh2, ow2] or NULL
 *  d_geom      : int32 [N,8] (x1,x2,y1,y2,new_h,new_w,y_off,x_off) or NULL
 *  max_box_h/w : host-side upper bound of the clipped box size (<= max delta sums); used
 *                to size shared memory.  SVB_ERR_BOX_TOO_LARGE if it cannot fit on chip.
 *  flags       : SVB_K3_NO_NORMALIZE = the slices already hold uint8 values (0..255 as float):
 *                skip the per-crop min-max and only cast -- resize_with_padding on uint8 input.
 */
#define SVB_K3_NO_NORMALIZE 1
#define SVB_K3_XY_F64 2
size_t svb_k3_workspace_bytes(int ch, int cw, int oh2, int ow2);
int svb_k3_crop_resample(const float* d_slices, const int64_t* d_offs, const int32_t* d_hw,
                         const int32_t* d_slice_idx, const float* d_xy, const int32_t* d_delta_px,
                         int N, int max_box_h, int max_box_w, int ch, int cw, uint8_t* d_crops,
                         int oh2, int ow2, uint8_t* d_crops2, int32_t* d_geom, int flags, void* d_ws,
                         size_t ws_bytes, void* stream);

/* Rotated crop mode (CropContext mode="rotated": crop_region_rotated, cropping.py:258-313): same as above, but the box is
 * cut from cv2.warpAffine(image, R, INTER_LINEAR, BORDER_REPLICATE) about the disc centre, evaluated on the fly.
 *  d_inv_affine : float64 [N,6] -- the INVERSE of cv2.getRotationMatrix2D((cx,cy), angle, 1.0) per crop, row-major 2x3,
 *                 computed on the host exactly as cv::warpAffine inverts it (spine_vision_b200.cropping.inverse_rotation);
 *                 NULL = horizontal mode.
 *  d_pixel_kind : int32 [B] per SLICE, or NULL (= all SVB_PIXEL_FLOAT): the pixel type the slice had in the file.  The
 *                 reference hands cv2.warpAffine the slice in that type (extract_middle_slice keeps it, cropping.py:63-79), so
 *                 int16 / uint16 sources are blended in fp32 and rounded back to the type (cvRound, saturating), uint8 sources
 *                 take OpenCV's 15-bit fixed-point path; the values still arrive here as float32. */
#define SVB_PIXEL_FLOAT 0
#define SVB_PIXEL_INT16 1
#define SVB_PIXEL_UINT16 2
#define SVB_PIXEL_UINT8 3
int svb_k3_crop_resample_rotated(const float* d_slices, const int64_t* d_offs, const int32_t* d_hw,
                                 const int32_t* d_slice_idx, const float* d_xy, const int32_t* d_delta_px,
                                 const double* d_inv_affine, const int32_t* d_pixel_kind, int N, int max_box_h,
                                 int max_box_w, int ch, int cw, uint8_t* d_crops, int oh2, int ow2, uint8_t* d_crops2,
                                 int32_t* d_geom, int flags, void* d_ws, size_t ws_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * K2 -- CoordinateRegressor forward (ConvNeXt backbone + MLP head + sigmoid).
 * Replaces model(tensor) in predict_ivd_locations (cropping.py:474-475) =
 * CoordinateRegressor.forward (spine_vision/training/models/generic.py:389-391) over the
 * timm convnext backbone made by BackboneFactory.create
 * (spine_vision/training/models/backbone.py:165-172) and the head at generic.py:343-351.
 *
 * svb_model_create takes the checkpoint's "model_state_dict" (load_localization_model,
 * cropping.py:436-437) as an array of HOST fp32 tensors under their state-dict names; it
 * folds /255 + ImageNet mean/std + RGB replication into the 4x4 stem, repacks the weights
 * for the tensor-core kernels and uploads them.  Supported: stage widths that are multiples of 32
 * in [96, 2816] and stem widths 96 / 128 / 192 / 256 / 352, i.e. every model_variant (tiny, small,
 * base, large, xlarge, v2_tiny .. v2_large, and v2_huge: 352 / 704 / 1408 / 2816); anything else is
 * SVB_ERR_UNSUPPORTED_MODEL.  With SVB_LN_FOLD=0 (the un-folded LayerNorm block) v2_huge is refused.
 */
typedef struct svb_model svb_model;

typedef struct svb_weight_desc {
    const char* name;    /* e.g. "backbone.stages.2.blocks.13.mlp.fc1.weight" */
    const float* data;   /* host, fp32, contiguous */
    int32_t ndim;
    int64_t shape[4];
} svb_weight_desc;

int svb_model_create(svb_model** out, const svb_weight_desc* weights, int n_weights, int dtype);
int svb_model_destroy(svb_model* m);
/* bytes of workspace svb_model_forward needs for micro-batches of `micro_batch` images.  By default this is TWO micro-batch
 * workspaces: svb_model_forward then keeps two micro-batches in flight -- even ones on the caller's stream, odd ones on a
 * stream the handle owns (created in svb_model_create), forked from and joined back into the caller's stream by events, so
 * the call stays asynchronous and ordered on `stream`.  SVB_DUAL_CHAIN=0 (or a workspace of half the size) keeps one. */
size_t svb_model_workspace_bytes(const svb_model* m, int micro_batch, int H, int W);
/*  d_in_u8  : uint8 [B, H, W] -- K1 output (one plane)
 *  d_coords : float32 [B, num_levels, 2] in [0,1]
 *  micro_batch : images per pass through the network (activation working set ~ L2-sized)
 *  d_times_ms : optional HOST float[SVB_NUM_KERNEL_CLASSES]; when non-NULL the call records
 *               CUDA events around every launch, synchronises at the end and accumulates
 *               per-kernel-class milliseconds (profiling / roofline only).
 */
enum { SVB_KC_STEM = 0, SVB_KC_DWCONV_LN = 1, SVB_KC_GEMM = 2, SVB_KC_LN_PATCHIFY = 3, SVB_KC_HEAD = 4, SVB_KC_MLP_FUSED = 5, SVB_NUM_KERNEL_CLASSES = 6 };
int svb_model_forward(svb_model* m, const uint8_t* d_in_u8, int B, int H, int W, float* d_coords,
                      int micro_batch, void* d_ws, size_t ws_bytes, void* stream, float* times_ms);
/* The same forward from the tensor the reference's callers build themselves: float32 NCHW [B,3,H,W], already /255 and
 * ImageNet-normalised (cropping.py:463-472) -- what `model(tensor)` receives (generic.py:389-391; notebooks,
 * BaseModel.test_inference base.py:153-158).  Un-folded stem conv (3 input channels); everything after the stem is the
 * same code.  The dataset path does not use it (it feeds K1's uint8 plane to the folded stem). */
int svb_model_forward_f32(svb_model* m, const float* d_in_nchw, int B, int H, int W, float* d_coords,
                          int micro_batch, void* d_ws, size_t ws_bytes, void* stream, float* times_ms);
/* svb_model_forward (same kernels, micro-batches, streams and plans) that also reads out the residual stream after the last
 * block of stages 0 .. n_stage_out - 1 (tests, profiling): d_stage_out[s] is a device buffer [B, H / 2^(s+2), W / 2^(s+2), dims[s]]
 * of the model dtype, written by one device-to-device copy per micro-batch on the stream that computed it.  1 <= n_stage_out <= 4. */
int svb_model_forward_stages(svb_model* m, const uint8_t* d_in_u8, int B, int H, int W, float* d_coords, int micro_batch,
                             void* d_ws, size_t ws_bytes, void* stream, void* const* d_stage_out, int n_stage_out);
/* CUDA graph of one svb_model_forward / svb_model_forward_f32: the same kernels, micro-batches, second chain, tail micro-batch,
 * programmatic dependent launches and clusters, captured once and replayed with one cudaGraphLaunch per call.
 *  create  : checks its arguments as svb_model_forward does, captures one forward over B images of H x W with `micro_batch` on
 *            `stream` (thread-local capture mode; not the legacy default stream, and not a stream that is already capturing)
 *            and instantiates it (allocating what the graph needs; nothing is enqueued on `stream`).  A capture that fails is ended and discarded: the call returns a negative svb_status and the
 *            stream stays usable.  input_kind: SVB_GRAPH_INPUT_U8 (uint8 [B,H,W] planes, folded stem) or SVB_GRAPH_INPUT_F32
 *            (float32 [B,3,H,W], as svb_model_forward_f32).
 *  launch  : d_in / d_coords may differ on every call (the nodes that read the input and write the coordinates are rebound; a
 *            replay already enqueued keeps its pointers).  Asynchronous on `stream`; adds the graph's kernel-node count to
 *            svb_launch_count.  Replays of one graph run one after another, whatever stream they are launched on.
 *  info    : out[0] = kernel nodes (the launches of one svb_model_forward with the same arguments), out[1..3] = B, H, W.
 * The graph binds d_ws for its lifetime and owns no workspace: the caller keeps it alive and does not use it for anything else
 * while the graph exists.  Destroy the graph before its model.  Shapes are fixed at capture: another B, H, W or micro-batch is
 * another graph.  Per-stage readout (svb_model_forward_stages) and per-launch timing (times_ms) are not supported in graphs; a
 * svb_model_forward / svb_model_forward_f32 on a stream that is capturing records correctly (torch.cuda.graph), but refuses
 * times_ms with SVB_ERR_INVALID_ARG.  A handle is not thread-safe, like svb_model. */
typedef struct svb_model_graph svb_model_graph;
#define SVB_GRAPH_INPUT_U8 0  /* svb_model_forward: uint8 [B,H,W] planes, folded stem */
#define SVB_GRAPH_INPUT_F32 1 /* svb_model_forward_f32: float32 [B,3,H,W], model(tensor) */
int svb_model_graph_create(svb_model* m, int input_kind, int B, int H, int W, int micro_batch, void* d_ws, size_t ws_bytes,
                           void* stream, svb_model_graph** out);
int svb_model_graph_launch(svb_model_graph* g, const void* d_in, float* d_coords, void* stream);
int svb_model_graph_info(const svb_model_graph* g, int32_t out[4]); /* kernel nodes, B, H, W */
int svb_model_graph_destroy(svb_model_graph* g);
/* model geometry: out[0]=num_levels, out[1]=num_outputs, out[2..5]=dims, out[6..9]=depths */
int svb_model_info(const svb_model* m, int32_t out[10]);
/* total tensor-core GEMM flops and launches of one forward over B images (for the roofline) */
int svb_model_cost(const svb_model* m, int B, int H, int W, double* gemm_flops, int64_t* launches);

/* Standalone GEMM entry for unit tests / ncu: D[M,N] = epilogue(A[M,K] * Wt[N,K]^T).
 * mode 0: out = gelu(acc + bias)            (fc1)
 * mode 1: out = resid + gamma*(acc + bias)  (fc2; resid may alias out)
 * mode 2: out = acc + bias                  (downsample conv as GEMM)
 * All matrices row-major 16-bit of `dtype`; bias/gamma fp32 [N]. */
int svb_gemm(const void* d_a, const void* d_w, void* d_out, const void* d_resid, const float* d_bias,
             const float* d_gamma, int M, int N, int K, int mode, int dtype, void* stream);

/* Standalone fused ConvNeXt MLP (unit tests / ncu): x <- x + gamma * (fc2(GELU(fc1(a) + b1)) + b2) in one kernel, the
 * hidden activation [M,4C] stays on chip.  a [M,C], w1 [4C,C], w2 [C,4C], x [M,C] (in place), 16-bit of `dtype`;
 * b1 [4C], b2 [C], gamma [C] fp32.  C = 128 or 256 (Y + two hidden accumulators must fit the 512 TMEM columns). */
int svb_mlp_fused(const void* d_a, const void* d_w1, const float* d_b1, const void* d_w2, const float* d_b2,
                  const float* d_gamma, void* d_x, int M, int C, int dtype, void* stream);
/* The same with the block's LayerNorm folded into fc1 (what the model runs at C = 128 / 256): d_a = the RAW depthwise output,
 * d_w1g = r16(W1 diag(g)), d_t / d_s / d_rowstat as svb_gemm mode 3's d_bias / d_gamma / d_resid. */
int svb_mlp_fused_ln(const void* d_a, const void* d_w1g, const float* d_t, const float* d_s, const float* d_rowstat, const void* d_w2,
                     const float* d_b2, const float* d_gamma, void* d_x, int M, int C, int dtype, void* stream);

/* ------------------------------------------------------------------------------------------
 * Standalone layer entries (unit tests / ncu captures of one kernel).  Same kernels the model runs.
 * x/out are NHWC 16-bit of `dtype`.
 *  svb_stem_ln     : u8 [B,H,W] -> [B,H/4,W/4,C0]; wf [C0][16], bf [C0] are the FOLDED stem (fp32); C0 = 96/128/192/256/352
 *  svb_dwconv_ln   : depthwise 7x7 (taps [49][C] fp32, tap-major) + bias + LayerNorm(C) eps 1e-6
 *  svb_ln_patchify : LayerNorm2d + 2x2/s2 gather -> [B,H/2,W/2,4C]; C = the stage-0..2 widths (96..1024, 352/704/1408)
 *  svb_head        : avg-pool over `tokens` + LayerNorm(eps 1e-6) + LayerNorm(eps 1e-5)
 *                    + Linear(C,HID) + GELU + Linear(HID,NOUT) + sigmoid -> coords fp32 [B,NOUT]
 */
int svb_stem_ln(const uint8_t* d_in, const float* d_wf, const float* d_bf, const float* d_lnw, const float* d_lnb,
                void* d_out, int B, int H, int W, int C0, int dtype, void* stream);
int svb_dwconv_ln(const void* d_x, const float* d_taps, const float* d_bias, const float* d_lnw,
                  const float* d_lnb, void* d_out, int B, int H, int W, int C, int dtype, void* stream);
/* Depthwise 7x7 + bias with the block's LayerNorm FOLDED INTO fc1 (the default forward): d_out = the raw convolution, 16-bit
 * [B,H,W,C] (fc1's A operand); d_rowstat = float32 [B*H*W, 2] = (rstd, -mean * rstd) of each token's C rounded values.  fc1 is
 * then svb_gemm(mode 3): GELU(rstd_m * (A @ (W1 diag(g))^T)[m,n] + (-mean_m rstd_m) * s_n + t_n), with d_w = r16(W1 * g),
 * d_gamma = s_n = sum_k r16(W1 g)[n,k], d_bias = t_n = W1 @ ln_bias + b1, d_resid = d_rowstat.
 * (timm ConvNeXt block: conv_dw -> norm -> mlp.fc1 -> act; generic.py:389-391 over backbone.py:165-172.) */
int svb_dwconv_raw(const void* d_x, const float* d_taps, const float* d_bias, void* d_out, float* d_rowstat, int B, int H, int W,
                   int C, int dtype, void* stream);

/* The same operator on the tensor cores (dwconv_rawtc_kernel: seven row-shifted tcgen05 MMAs per 16 channels with the stencil
 * columns side by side in N, column sum by warp shuffles; DESIGN.md section 4); what the model runs for fp16.  Same outputs as
 * svb_dwconv_raw (d_out, d_rowstat); the taps are 16-bit operands: d_wtc = svb_dwconv_tc_pack(taps) ([C/64][7][112][64] of
 * `dtype`, packed on the HOST from fp32 [49][C]).  d_stat_part = scratch, float32 [B*H*W][C/64][2] (each token's sum / sum of
 * squares per 64-channel chunk; a second small launch adds them up into d_rowstat).  C must be a multiple of 64. */
int svb_dwconv_tc_pack(const float* h_taps, void* h_wtc, int C, int dtype);
int svb_dwconv_raw_tc(const void* d_x, const void* d_wtc, const float* d_bias, void* d_out, float* d_rowstat, float* d_stat_part, int B,
                      int H, int W, int C, int dtype, void* stream);

int svb_ln_patchify(const void* d_x, const float* d_lnw, const float* d_lnb, void* d_out, int B, int H, int W,
                    int C, int dtype, void* stream);
int svb_head(const void* d_x, int B, int tokens, int C, const float* n0w, const float* n0b, const float* n1w,
             const float* n1b, const float* w1, const float* b1, int HID, const float* w2, const float* b2,
             int NOUT, float* d_coords, int dtype, void* stream);

/* ------------------------------------------------------------------------------------------
 * K4 -- classifier-input producer (SURVEY.md 8(f) row 4).
 * Replaces, for a batch of (patient, level) samples, construct_3channel + transforms.Resize + ToTensor + Normalize of
 * ClassificationDataset (spine_vision/training/datasets/classification.py:40-68, 247-278, 283-304; no augmentation):
 * Pillow resizes each band on its own, so the resized bands are K3's second output and this call is the
 * [T2, T1, T2] stack (one series three times when the other is missing) + /255 + (x - mean) / std, with torch's fp32
 * operation order (bit-exact for float32 output).
 *  d_planes   : uint8 [N, H, W]   resized crops (K3 second output)
 *  d_t2_idx, d_t1_idx : int32 [P] plane index of each sample's T2 / T1 crop, -1 = the series is missing
 *               (both -1: the sample is left untouched; the reference raises ValueError, so does the Python mirror)
 *  h_mean3, h_std3 : HOST float[3], NULL = ImageNet (classification.py:270-273); normalize = 0 skips Normalize
 *  out_dtype  : SVB_F32 (reference), SVB_BF16 or SVB_FP16 (rounded from the fp32 value)
 *  d_out      : [P, 3, H, W] of out_dtype
 */
int svb_k4_classifier_input(const uint8_t* d_planes, const int32_t* d_t2_idx, const int32_t* d_t1_idx, int P, int H,
                            int W, const float* h_mean3, const float* h_std3, int normalize, int out_dtype,
                            void* d_out, void* stream);

/* ------------------------------------------------------------------------------------------
 * Host input / output stage (SURVEY.md 8(f) row 3): plain host code, no CUDA; h_* are HOST pointers.
 *
 * PNG -- replaces Image.fromarray(crop).save(path) (datasets/classification/spider.py:158, phenikaa.py:213):
 * 8-bit greyscale (PIL mode "L"), non-interlaced, zlib `level` (Pillow's default is 6; out of range = 6), adaptive row
 * filters.  Parity is on the decoded pixels.  The batch call encodes and writes with `n_threads` workers
 * (<= 0: one per hardware thread); rcs (optional, [n]) receives the per-file status.
 */
size_t svb_png_bound(int h, int w); /* bytes svb_png_encode_gray8 may need for one image */
int svb_png_encode_gray8(const uint8_t* h_img, int h, int w, int level, uint8_t* h_out, size_t cap, size_t* out_len);
int svb_png_write_gray8_batch(const uint8_t* h_imgs /* [n, h, w] */, int n, int h, int w, const char* const* paths,
                              int level, int n_threads, int32_t* rcs);
/* images of different sizes: image i = hw[2i] x hw[2i+1] bytes at h_pool + offs[i] */
int svb_png_write_gray8_ragged(const uint8_t* h_pool, const int64_t* offs, const int32_t* hw, int n, const char* const* paths,
                               int level, int n_threads, int32_t* rcs);

/* MetaImage (.mha, .mhd + raw / zraw) -- replaces read_medical_image -> read_mha -> sitk.ReadImage for the SPIDER
 * volumes (spine_vision/io/readers.py:65-73, 128-161; spider.py:115).  Scalar 2-D / 3-D images, binary data, raw or
 * zlib-compressed, either byte order.  Voxels are converted to float32 in file order = sitk.GetArrayFromImage order
 * [z][y][x] (integer types up to 24 bits and float32 exactly; wider types are rounded to float32).
 * direction is image.GetDirection() (row-major 3x3: COLUMN a = direction cosine of image axis a, i.e. the transpose of
 * the file's TransformMatrix), spacing = GetSpacing(), origin = GetOrigin(), dim = GetSize() (x, y, z).
 */
typedef enum svb_mha_type {
    SVB_MHA_I8 = 0, SVB_MHA_U8 = 1, SVB_MHA_I16 = 2, SVB_MHA_U16 = 3, SVB_MHA_I32 = 4, SVB_MHA_U32 = 5,
    SVB_MHA_I64 = 6, SVB_MHA_U64 = 7, SVB_MHA_F32 = 8, SVB_MHA_F64 = 9
} svb_mha_type;
typedef struct svb_mha_info {
    int32_t ndim;
    int32_t dim[3];            /* x, y, z (1 beyond ndim) */
    double spacing[3];
    double origin[3];
    double direction[9];
    int32_t element_type;      /* svb_mha_type */
    int32_t element_bytes;
    int32_t channels;
    int32_t compressed;
    int32_t big_endian;
    int32_t has_spacing;       /* ElementSpacing was given (else ElementSize or 1.0) */
    int64_t data_offset;       /* byte offset of the voxel data in the header file (ElementDataFile = LOCAL), else -1 */
    int64_t header_size;       /* HeaderSize of a separate data file (-1 = data at the end of the file) */
    int64_t compressed_size;   /* CompressedDataSize, 0 = to the end of the file */
    char data_file[1024];      /* separate data file (resolved against the header's directory), "" when LOCAL */
} svb_mha_info;
int svb_mha_read_header(const char* path, svb_mha_info* info);
int svb_mha_read_f32(const char* path, const svb_mha_info* info, float* h_dst, size_t dst_elems);
/* n volumes on n_threads workers into caller-owned (pinned) buffers; rcs (optional, [n]) = per-file status, so that the
 * caller can skip unreadable series the way the reference's drivers do (spider.py:139-141). */
int svb_mha_read_batch_f32(const char* const* paths, int n, const svb_mha_info* infos, float* const* h_dsts,
                           const size_t* dst_elems, int n_threads, int32_t* rcs);

/* Slices [z0[i], z1[i]) of volume i only, written at their place in the buffer of the WHOLE volume (h_dsts[i], dst_elems[i] as
 * above; the rest of the buffer is not touched).  The dataset driver needs the two source slices around the middle sagittal
 * plane (cropping.py:63-79 keeps one plane of the resampled volume): a zlib stream is inflated up to the slab and no further,
 * only the slab is converted to float32. */
int svb_mha_read_batch_slab_f32(const char* const* paths, int n, const svb_mha_info* infos, float* const* h_dsts,
                                const size_t* dst_elems, const int32_t* z0, const int32_t* z1, int n_threads, int32_t* rcs);

/* DICOM series (one slice per file) -- replaces read_medical_image -> read_dicom_series -> sitk.ImageSeriesReader over
 * GDCM for the Phenikaa series directories (spine_vision/io/readers.py:48-73, 128-161; phenikaa.py:178).  Part-10 files,
 * implicit / explicit VR little endian or explicit big endian with native pixel data, and the two lossless ENCAPSULATED
 * transfer syntaxes MR exports use: RLE Lossless (1.2.840.10008.1.2.5, PS3.5 Annex G) and JPEG Lossless, process 14
 * (1.2.840.10008.1.2.4.57 and .70: ITU-T T.81 Annex H, Huffman, predictors 1-7, restart intervals); GDCM decodes both for
 * the reference.  Lossy JPEG, JPEG-LS and JPEG 2000 give SVB_ERR_FORMAT.  Monochrome 8 / 16 / 32 bit; BitsStored <
 * BitsAllocated is masked / sign-extended like GDCM does; MONOCHROME1 gives SVB_ERR_FORMAT (ITK inverts it to MONOCHROME2:
 * never decoded un-inverted behind the caller's back).  The C side parses and decodes single files on a thread pool; series
 * selection, slice ordering and the volume geometry (the ITK conventions) are host logic in spine_vision_b200/hostio.py.
 * Parity is UNPINNED (SimpleITK / GDCM are absent from the build image; restated in oracle/dicom.py).
 */
typedef struct svb_dicom_info {
    int32_t rows, cols, bits_allocated, pixel_representation, samples_per_pixel, monochrome1;
    int32_t instance_number, big_endian, has_position, has_orientation, has_spacing;
    int32_t encapsulation;          /* SVB_DICOM_NATIVE / _RLE / _JPEG_LOSSLESS: how (7FE0,0010) is stored */
    double pixel_spacing[2];        /* (0028,0030): row spacing (between rows), column spacing */
    double position[3];             /* (0020,0032) ImagePositionPatient */
    double orientation[6];          /* (0020,0037) ImageOrientationPatient: row cosines, column cosines */
    double rescale_slope, rescale_intercept; /* (0028,1053), (0028,1052); applied by svb_dicom_read_slices_f32 */
    double slice_thickness, spacing_between_slices;
    int64_t pixel_offset, pixel_bytes; /* (7FE0,0010): native = the samples; encapsulated = the first item .. end of file */
    int32_t bits_stored, pad;       /* (0028,0101) */
    char series_uid[72];            /* (0020,000E) */
} svb_dicom_info;
#define SVB_DICOM_NATIVE 0
#define SVB_DICOM_RLE 1
#define SVB_DICOM_JPEG_LOSSLESS 2
/* rcs (optional, [n]) = per-file status: files that are not (supported) DICOM are dropped by the caller */
int svb_dicom_read_headers(const char* const* paths, int n, svb_dicom_info* infos, int n_threads, int32_t* rcs);
/* slice i -> h_dsts[i] (rows*cols float32, stored value * slope + intercept), on n_threads workers */
int svb_dicom_read_slices_f32(const char* const* paths, int n, const svb_dicom_info* infos, float* const* h_dsts,
                              const size_t* dst_elems, int n_threads, int32_t* rcs);

#ifdef __cplusplus
}
#endif
#endif /* SPINE_B200_H_ */
