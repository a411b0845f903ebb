/* codenet_b200 -- C ABI of the B200-native CoDeNet inference hot path (libcodenet_b200.so).
 *
 * Plain pointers and sizes only; every function returns 0 on success or a negative cdn_status, and
 * cdn_last_error() returns a thread-local message.  No exception crosses this boundary, no hidden device
 * allocation happens after cdn_engine_finalize(), all device pointers are caller-owned unless stated, and every
 * launch goes to the cudaStream_t passed in (the reference launches on the legacy default stream and only
 * printf()s launch errors, lib/models/external/src/dcn_deform_conv_cuda_kernel.cu:264-275).
 *
 * Reference interfaces replaced (paths relative to the reference tree, see INTEGRATION.md for the bindings):
 *   cdn_deform_conv_forward_f32   <- deform_conv_forward_cuda, lib/models/external/src/dcn_deform_conv_cuda.cpp:151-258
 *                                    (pybind export :681-695; called from functions/dcn_deform_conv.py:51-56)
 *   cdn_deform_dw_w4a8            <- QuantDeformConvWithOffsetScaleBoundPositive.forward up to quant_identity_deform,
 *                                    portable_quantizer/quant_modules.py:668-671 (scale conv :648-650, Hardtanh+QuantAct
 *                                    :651-653, QuantDeformConv2d :473-517, QuantAct :202-225)
 *   cdn_pw_gemm_i8                <- QuantBnConv2d.forward / Quant_Conv2d.forward for 1x1 convs, quant_modules.py:364-419,
 *                                    :278-321, with the following ReLU + QuantAct and cat/channel_shuffle
 *                                    (lib/models/networks/shufflenetv2_dcn.py:29-34) folded into the store
 *   cdn_dw3x3_i8                  <- QuantBnConv2d.forward for depthwise 3x3 convs (same lines) + QuantAct
 *   cdn_stem_f32_i8               <- layer0 = QuantBnConv2d(8 bit) + ReLU + QuantAct [+ MaxPool], quantize_model.py:26-35
 *   cdn_ctdet_decode              <- ctdet_decode, lib/models/decode.py:474-505 (_nms :10-16, _topk :110-126)
 *   cdn_ctdet_merge               <- CtdetDetector.merge_outputs, lib/detectors/ctdet.py:59-74 (with post_process's division by the
 *                                    scale, base_detector.py post_process)
 *   cdn_soft_nms                  <- soft_nms, lib/models/external/nms.pyx:77-170
 *   cdn_engine_*                  <- PoseShuffleNetV2.forward (shufflenetv2_dcn.py:314-330) as rewritten by
 *                                    quantize_shufflenetv2_dcn (quantize_model.py:7-82) + CtdetDetector.process
 *                                    (lib/detectors/ctdet.py:29-46)
 *
 * Activation layout: NHWC int8, `pitch` bytes per pixel (a multiple of 32); the real value of an element is
 * (q + z) / s for the (s, z) of the QuantAct that produced it (quant_utils.py:58-73).
 *
 * Requantisation constants (one per output channel, see DESIGN.md): q = clamp(rint(acc*M + B), lo, 127) with
 * M, B in fp64.  The library solves, per channel, for an exact 64-bit fixed-point form of this step function
 * (cdn_rq_int_solve); where none exists it derives an fp32 copy and a guard band inside which the kernels re-evaluate in
 * fp64.  Either way results are bit-identical to the fp64 formula.
 */
#ifndef CODENET_B200_H
#define CODENET_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* cdn_stream_t;                 /* a cudaStream_t */

typedef enum {
  CDN_OK = 0,
  CDN_ERR_INVALID = -1,                     /* bad argument / unsupported shape */
  CDN_ERR_CUDA = -2,                        /* CUDA runtime or driver error (message has the CUDA string) */
  CDN_ERR_NO_DEVICE = -3,                   /* no usable sm_100 device: there is NO CPU fallback */
  CDN_ERR_STATE = -4                        /* engine used in the wrong order */
} cdn_status;

const char* cdn_last_error(void);
int cdn_version(void);
/* 0 = ok; CDN_ERR_NO_DEVICE if `device` is not a compute-capability-10.x GPU. */
int cdn_check_device(int device);
/* Bring-up / measurement switches, never needed in production.  bit 0: 1x1 convolutions on the SIMT cross-check kernel
 * instead of tcgen05; bit 1: no CUDA graph (eager launches); bit 4: in-kernel phase cycle accounting of the GEMM
 * (tools/pw_phase_cycles.py); bit 6: no programmatic dependent launch; bit 7 (read when a layer is built): guarded fp32
 * requantisation instead of the integer form (same results, A/B timing); bit 8: never fuse the heads' tail (as option
 * "fuse_heads" = 0); bit 9: depthwise convs on the LDG kernel instead of the TMA-staged one, bit 10: the stride-2 ones only
 * (same results, A/B timing); bits 2, 3, 5: experiments that BREAK results. */
int cdn_set_debug_flags(unsigned flags);

/* ---- per-output-channel requantisation constants (host arrays, length n) ------------------------------- */
typedef struct {
  const double* M;                          /* s_out / (sigma_c * s_x) */
  const double* B;                          /* s_out * b'_c - z_out */
  int lo;                                   /* max(-128, relu ? -z_out : -128) */
  int n;
} cdn_requant;

/* Host-only helper (no device needed): the fixed-point form the int8 kernels evaluate,
 *   q = sat8(max((((int64)v*Mi + Bi) >> 32) >> sh, lo)),
 * solved so that it equals clamp(rint(fl64(fl64(v*M) + B)), lo, 127) for EVERY integer accumulator v in [vmin, vmax]
 * (DESIGN.md "requantisation").  Returns CDN_ERR_INVALID when no exact pair exists (M >= 0.5 or M <= 0); layers fall back
 * to the guarded fp32 sequence in that case.  Exposed so the exactness claim can be tested exhaustively on the CPU. */
int cdn_rq_int_solve(double M, double B, int lo, int64_t vmin, int64_t vmax, int32_t* Mi, int32_t* sh, int64_t* Bi);

/* ---- stem: fp32 NCHW image -> int8 NHWC -----------------------------------------------------------------
 * 3x3 conv, pad 1, stride `stride`, 3 -> C (C <= 32), 8-bit integer weights wq[C][3][3][3] (host), then ReLU and
 * QuantAct.  If pool != 0 a MaxPool2d(3,2,1) follows on the quantised grid.  out pitch = 32. */
int cdn_stem_f32_i8(const float* d_img, int batch, int H, int W, int stride, int pool,
                    const int8_t* wq, int C, const cdn_requant* rq, int8_t* d_out, int out_pitch,
                    cdn_stream_t stream);

/* ---- depthwise 3x3 (pad 1), int8 NHWC -> int8 NHWC -------------------------------------------------------
 * wq[C][9] (host).  in_shift = 1 reads the input through a virtual nearest x2 upsample (input stored at H/2 x W/2).
 * zx is the input zero point: out-of-image taps contribute real zero, i.e. q = -zx, which must fit int8. */
int cdn_dw3x3_i8(const int8_t* d_in, int in_pitch, int batch, int H, int W, int in_shift, int stride,
                 const int8_t* wq, int C, int zx, const cdn_requant* rq, int8_t* d_out, int out_pitch,
                 cdn_stream_t stream);

/* ---- fused co-designed deformable depthwise conv (W4A8) --------------------------------------------------
 * Per output pixel: u = clamp(acc_s*Ms + bs, -bound+1, bound) with acc_s = sum_c ws[c]*(q+zx);
 * qs = rint(ss*u - zs); s = (qs+zs)/ss; mode 0: s = rint(s) and tap (i,j) reads pixel (h+(i-1)s, w+(j-1)s);
 * mode 1: bilinear sampling at the fractional position (reference default).  Then 3x3 depthwise MAC with wq[C][9]
 * and requantisation.  H, W are the OUTPUT/sampling-grid size; in_shift as for cdn_dw3x3_i8.
 * d_sval (optional, may be NULL): float [batch*H*W] receives s as used. */
typedef struct {
  const int8_t* ws;                         /* [C] 4-bit integer weights of the C->1 scale conv (host) */
  double Ms, bs;                            /* 1/(sigma_s*s_x), bias */
  double ss, zs;                            /* QuantAct of s */
  int bound;                                /* offset_bound (Hardtanh -bound+1 .. bound) */
  int mode;                                 /* 0 = integer offsets (round half even), 1 = bilinear */
} cdn_deform_scale;

int cdn_deform_dw_w4a8(const int8_t* d_in, int in_pitch, int batch, int H, int W, int in_shift,
                       const cdn_deform_scale* sc, const int8_t* wq, int C, int zx, const cdn_requant* rq,
                       int8_t* d_out, int out_pitch, float* d_sval, cdn_stream_t stream);

/* The same layer with its constants uploaded once (no allocation or synchronisation per call): what an integration that
 * keeps the reference's module structure holds per QuantDeformConvWithOffsetScaleBoundPositive, and what the isolated
 * layer sweep (tools/deform_sweep.py, BASELINE config 2) times.  `pitch` = bytes per pixel of the tensors it will see. */
typedef struct cdn_deform_layer cdn_deform_layer;
int cdn_deform_layer_create(cdn_deform_layer** out, const cdn_deform_scale* sc, const int8_t* wq, int C, int pitch, int zx,
                            const cdn_requant* rq);
int cdn_deform_layer_run(cdn_deform_layer* layer, const int8_t* d_in, int in_pitch, int batch, int H, int W, int in_shift,
                         int8_t* d_out, int out_pitch, float* d_sval, cdn_stream_t stream);
int cdn_deform_layer_destroy(cdn_deform_layer* layer);

/* ---- the steps either side of the path, on the device (SURVEY.md 8(f) rows 1-2) -----------------------------------
 * cdn_warp_affine_u8: cv2.warpAffine(image, M, (dst_w, dst_h), flags=cv2.INTER_LINEAR) of BaseDetector.pre_process
 * (lib/detectors/base_detector.py:61-65) on a uint8 HWC image [H][W][3], bit-identical to OpenCV (M6 = the 2x3 source ->
 * destination matrix cv2 receives, row-major doubles on the HOST); flip_copy != 0 also writes the mirrored image behind
 * the first one (dst [2][dst_h][dst_w][3], what --flip_test concatenates, :69-70).
 * cdn_ctdet_group_by_class: the grouping of ctdet_post_process (lib/utils/post_process.py:86-103): d_out [B][K][6] = the
 * detections ordered by class, original (score) order inside a class; d_counts [B][num_classes]. */
int cdn_warp_affine_u8(const uint8_t* d_src, int H, int W, const double* M6, uint8_t* d_dst, int dst_h, int dst_w, int flip_copy,
                       cdn_stream_t stream);

/* cdn_warp_affine_u8_batch: the same warpAffine for a ragged batch in one launch.  d_pool is a device byte pool holding source
 * frames of any sizes back to back (uint8 HWC [src_h][src_w][3] at src_offset, any byte offset); h_desc[n] is a HOST array with
 * one descriptor per output image: slot dst_slot of d_dst [dst_slots][dst_h][dst_w][3] receives
 * cv2.warpAffine(frame, M, (dst_w, dst_h), flags=cv2.INTER_LINEAR) bit for bit, and slot mirror_slot (-1 = none) its mirror
 * image (--flip_test).  Every argument is checked on the host before anything is launched (null pointers, n < 0, non-positive
 * sizes, a negative offset, slots outside [0, dst_slots)).  The matrices are inverted on the host and the descriptors travel as
 * kernel parameters (up to CDN_WARP_DESC_PER_LAUNCH per launch, more descriptors take several launches): no workspace, no
 * allocation, no synchronisation, so the call can be captured into a CUDA graph.  Slots no descriptor names are left as they
 * are.  cdn_warp_affine_u8 is the one-descriptor call {0, H, W, M6, 0, flip_copy ? 1 : -1} with dst_slots = 1 + flip_copy. */
typedef struct cdn_warp_desc {
  long long src_offset;              /* byte offset of the source frame in d_pool */
  int src_h, src_w;
  double M[6];                       /* the 2x3 source -> destination matrix cv2.warpAffine receives, row major */
  int dst_slot, mirror_slot;
} cdn_warp_desc;
#define CDN_WARP_DESC_PER_LAUNCH 454
int cdn_warp_affine_u8_batch(const uint8_t* d_pool, const cdn_warp_desc* h_desc, int n, uint8_t* d_dst, int dst_slots, int dst_h,
                             int dst_w, cdn_stream_t stream);

/* cdn_warp_affine_u8_f32_batch: the same ragged warp for the unquantised model, normalised into fp32 NCHW.  d_pool and h_desc as
 * for cdn_warp_affine_u8_batch; d_tables is a device array [n_tables][3][256] fp32 (n_tables 1 or 2) and h_table[n] a HOST
 * array with the table index of every descriptor.  Element (slot, c, y, x) of d_dst [dst_slots][3][dst_h][dst_w] is
 * table[h_table[i]][c][v], v the byte cdn_warp_affine_u8_batch writes at (slot, y, x, c), mirror slot included; channels keep
 * the frame's order.  The checks of cdn_warp_affine_u8_batch plus the tables pointer, n_tables and every table index, all on
 * the host before anything is launched; d_tables and d_dst 4-byte aligned (float4 stores when dst_w % 4 == 0 and d_dst is
 * 16-byte aligned).  No workspace, allocation or synchronisation: the call can be captured.  Up to
 * CDN_WARP_F32_DESC_PER_LAUNCH descriptors per launch. */
#define CDN_WARP_F32_DESC_PER_LAUNCH 448
int cdn_warp_affine_u8_f32_batch(const uint8_t* d_pool, const cdn_warp_desc* h_desc, const int32_t* h_table, int n,
                                 const float* d_tables, int n_tables, float* d_dst, int dst_slots, int dst_h, int dst_w,
                                 cdn_stream_t stream);
int cdn_ctdet_group_by_class(const float* d_dets, int batch, int K, int num_classes, float* d_out, int32_t* d_counts,
                             cdn_stream_t stream);

/* ---- baseline JPEG decoding on the device (csrc/jpeg.cu, DESIGN.md section 9) -------------------------------------------
 * cdn_jpeg_parse (HOST only, needs no device) reads the marker segments of one encoded image of nbytes bytes and fills *out.
 * Returns 0 when the device decodes the stream, a positive CDN_JPEG_HOST_* reason when only a host decoder does (the caller
 * decodes it with cv2.imdecode), or a negative CDN_JPEG_ERR_* when it is not a parseable JPEG.  Every read is bounded by
 * nbytes and every table is checked: malformed input returns a status.  The device takes SOF0/SOF1 8-bit, gray or YCbCr (the
 * libjpeg colour-space rule) with luma sampling 1x1, 2x1 or 2x2 and chroma 1x1, one interleaved scan holding every component,
 * 8- or 16-bit quantisation tables, any restart interval, and no Exif orientation other than 1.
 *
 * cdn_jpeg_decode_batch decodes n parsed frames in one call on `stream`: what cv2.imdecode(buf, cv2.IMREAD_COLOR) returns,
 * element for element, as uint8 BGR HWC [height][width][3] at out_offset of d_out (the source format of
 * cdn_warp_affine_u8_batch).  h_frames is the HOST array the caller filled (cdn_jpeg_parse, then data_offset, out_offset,
 * ws_offset) and d_frames a device copy of the same n descriptors, complete before the work on `stream` runs.  Stream i lies at
 * d_pool[data_offset, data_offset + nbytes); its workspace (restart offsets, int16 coefficient blocks, component planes) at
 * d_ws[ws_offset, ws_offset + ws_bytes), 256-byte aligned.  Every descriptor is checked on the host against pool_bytes,
 * ws_bytes and out_bytes first; then four kernels run (restart-marker index, entropy decode, dequantise + islow IDCT,
 * upsample + colour).  No allocation and no synchronisation: the call can be captured.  d_status[i] receives 0 when frame i
 * decoded, else CDN_JPEG_BAD_* bits: its output bytes are then undefined and the frame must be decoded on the host. */
#define CDN_JPEG_HOST_PROCESS 1        /* progressive, lossless, hierarchical or arithmetic-coded */
#define CDN_JPEG_HOST_PRECISION 2      /* not 8-bit samples */
#define CDN_JPEG_HOST_COLOR 3          /* neither 1 component nor 3 in YCbCr (CMYK, YCCK, RGB) */
#define CDN_JPEG_HOST_SAMPLING 4       /* 3 components other than 4:4:4, 4:2:2 or 4:2:0 */
#define CDN_JPEG_HOST_SCAN 5           /* several scans, a scan without every component, DNL, undefined tables */
#define CDN_JPEG_HOST_ORIENTATION 6    /* an Exif orientation other than 1 (cv2 rotates), or an Exif block it cannot read */
#define CDN_JPEG_HOST_SIZE 7           /* more than 2^26 pixels, or a stream of 2 GB or more */
#define CDN_JPEG_ERR_NOT_JPEG (-1)     /* no SOI marker */
#define CDN_JPEG_ERR_TRUNCATED (-2)    /* the headers end before the scan */
#define CDN_JPEG_ERR_SEGMENT (-3)      /* a marker segment with an impossible length or content */
#define CDN_JPEG_ERR_TABLE (-4)        /* a quantisation or Huffman table libjpeg rejects */
#define CDN_JPEG_BAD_CODE 1            /* an invalid Huffman code or a run past coefficient 63 */
#define CDN_JPEG_BAD_END 2             /* the data of a restart interval ends (marker or end of scan) before its last MCU */
#define CDN_JPEG_BAD_RESTART 4         /* restart markers missing, extra or out of sequence */
#define CDN_JPEG_BAD_RANGE 8           /* coefficients or IDCT outputs outside the window where libjpeg-turbo's C and SIMD agree */
#define CDN_JPEG_LOOKAHEAD 8

typedef struct cdn_jpeg_huff {         /* jpeg_make_d_derived_tbl's decoding form of one Huffman table */
  int32_t maxcode[18];                 /* largest code of each length 1..16, -1 if none; maxcode[17] = 0xFFFFF */
  int32_t valoffset[18];               /* huffval index of a code of length l = code + valoffset[l] */
  uint16_t look[1 << CDN_JPEG_LOOKAHEAD];  /* next 8 bits -> (length << 8) | symbol, 0 when the code is longer */
  uint8_t huffval[256];
} cdn_jpeg_huff;

typedef struct cdn_jpeg_frame {
  /* filled by cdn_jpeg_parse */
  int32_t width, height, ncomp;        /* ncomp 1 (gray) or 3 (YCbCr) */
  int32_t hmax, vmax;                  /* luma sampling factors (1 for gray) */
  int32_t mcux, mcuy;                  /* MCU grid */
  int32_t restart_interval;            /* MCUs per entropy-coded segment, 0 = none */
  int32_t nsegments;                   /* entropy-coded segments (restart intervals) */
  int32_t pad0;
  int64_t nbytes;                      /* bytes of the stream */
  int64_t scan_offset, scan_end;       /* entropy-coded bytes [scan_offset, scan_end) of the stream */
  int32_t comp_h[3], comp_v[3];        /* blocks per MCU of each component */
  int32_t comp_bw[3], comp_bh[3];      /* block grid of each component */
  int32_t comp_dw[3], comp_dh[3];      /* downsampled (valid) size of each component */
  int32_t comp_dc[3], comp_ac[3];      /* Huffman table of each component: huff[0..1] DC, huff[2..3] AC */
  int64_t ws_bytes;                    /* workspace this frame needs */
  int64_t coef_rel, plane_rel[3];      /* workspace layout: restart offsets at 0, coefficients, planes */
  uint16_t qt[3][64];                  /* dequantisation table of each component, natural order */
  cdn_jpeg_huff huff[4];
  /* filled by the caller */
  int64_t data_offset;                 /* stream position in d_pool */
  int64_t out_offset;                  /* BGR frame position in d_out */
  int64_t ws_offset;                   /* workspace position in d_ws (a multiple of 256) */
} cdn_jpeg_frame;

int cdn_jpeg_parse(const uint8_t* data, int64_t nbytes, cdn_jpeg_frame* out);
int cdn_jpeg_decode_batch(const uint8_t* d_pool, int64_t pool_bytes, const cdn_jpeg_frame* h_frames,
                          const cdn_jpeg_frame* d_frames, int n, uint8_t* d_ws, int64_t ws_bytes, uint8_t* d_out,
                          int64_t out_bytes, int32_t* d_status, cdn_stream_t stream);

/* ---- multi-scale merge and soft-NMS (lib/detectors/ctdet.py:59-74, lib/models/external/nms.pyx:77-170) ---------------
 * cdn_soft_nms: the reference's soft_nms on n_seg independent segments of d_boxes [rows][5] (x1, y1, x2, y2, score), segment g =
 * rows [d_seg_off[g], d_seg_off[g+1]) (device int32, non-overlapping), each modified IN PLACE exactly as compat.soft_nms
 * modifies its array: the outer loop over the original length, the first maximum with row i winning ties, a discarded row
 * overwritten by a copy of row N-1, rows past the final N holding stale copies with their scores from before the pass.
 * d_keep[g] = the final N (what len(soft_nms(...)) returns).  method 0 hard, 1 linear, 2 gaussian.  Bit-identical to the mirror
 * (float / double sequence of compat/nms.py:40-53, exp = CUDA's double exp rounded to float).  max_len is the caller's bound on
 * the segment lengths; max_len > CDN_SOFT_NMS_MAX_LEN is CDN_ERR_INVALID before anything is launched, and a segment longer than
 * max_len (or with a negative start or length) is left untouched with d_keep = -1.  Scores must not be NaN.  Asynchronous.
 * cdn_ctdet_merge: CtdetDetector.merge_outputs (ctdet.py:59-74) for `batch` images with `scales` test scales each.  Inputs are
 * the outputs of cdn_ctdet_post_affine + cdn_ctdet_group_by_class for batch * scales network images, image-major and
 * scale-minor: d_grouped [batch*scales][K][6], d_counts [batch*scales][num_classes]; h_scales [scales] (host) the divisors of
 * post_process (base_detector.py post_process: coordinates / scale as a float32 division).  Per image and class the rows of
 * scale 0, 1, ... in grouped order (np.vstack order), coordinates divided by the scale; when scales > 1 or nms != 0 soft-NMS
 * per class with Nt 0.5, method 2, sigma 0.5, threshold 0.001, every row kept, stale tail included; then, if more than
 * max_per_image rows remain, only rows scoring >= the max_per_image-th largest score (np.partition) survive, in their order
 * (ties at the cut can keep more).  Outputs: d_rows [batch][scales*K][5] rows grouped by class (only the first
 * sum(d_class_counts[b]) rows of an image are written), d_class_counts [batch][num_classes].  Needs scales*K <=
 * CDN_SOFT_NMS_MAX_LEN, scales <= CDN_MERGE_MAX_SCALES, num_classes <= CDN_MERGE_MAX_CLASSES (CDN_ERR_INVALID otherwise,
 * checked on the host); one CTA per image keeps every intermediate in shared memory, so there is no workspace, no allocation
 * and no synchronisation: the call only enqueues one kernel on `stream`. */
#define CDN_SOFT_NMS_MAX_LEN 1024
#define CDN_MERGE_MAX_SCALES 16
#define CDN_MERGE_MAX_CLASSES 1024
int cdn_soft_nms(float* d_boxes, const int32_t* d_seg_off, int n_seg, int max_len, float sigma, float Nt, float threshold, int method,
                 int32_t* d_keep, cdn_stream_t stream);
int cdn_ctdet_merge(const float* d_grouped, const int32_t* d_counts, int batch, int scales, int K, int num_classes,
                    const float* h_scales, int nms, int max_per_image, float* d_rows, int32_t* d_class_counts, cdn_stream_t stream);

/* ---- module-level helpers: QuantAct on a real-valued tensor, MaxPool on the int8 grid -----------------------------
 * What compat.QuantAct.forward (portable_quantizer/quant_modules.py:202-225, frozen range) runs when it is handed an fp32
 * NCHW tensor: q = rint(fl64(fl64(scale*x) - zero)) (quant_utils.py:31-39) saturated to int8, written as int8 NHWC with
 * `out_pitch` bytes per pixel.  cdn_maxpool3s2_i8: nn.MaxPool2d(3, 2, 1) of an int8 NHWC grid (quantize_model.py:31-35). */
int cdn_quantize_f32_i8(const float* d_in, int batch, int C, int H, int W, double scale, double zero, int8_t* d_out,
                        int out_pitch, cdn_stream_t stream);
int cdn_maxpool3s2_i8(const int8_t* d_in, int batch, int H, int W, int pitch, int8_t* d_out, cdn_stream_t stream);

/* ---- 1x1 convolution as int8 tcgen05 GEMM ---------------------------------------------------------------
 * acc[p][n] = sum_k wq[n][k] * (in[p][k_off + k] + zx)   (exact int32; the library adds zx*sum_k wq[n][k] itself)
 * Output "chunks" describe where each group of <=16 output channels lands in the NHWC row, so that split /
 * cat / channel_shuffle cost nothing: a chunk takes `count` consecutive GEMM columns starting at `col`, optionally
 * interleaves them with `count` bytes of a pass-through tensor starting at byte `pass_off` (out[2i] = pass[i],
 * out[2i+1] = new[i]), zero-fills up to 16 bytes and stores them at byte `dst_off` of the output pixel. */
typedef struct {
  int16_t col;                              /* first GEMM column (multiple of 8) */
  int16_t count;                            /* valid columns: <=16 plain, <=8 interleaved, 0 = zero fill */
  int16_t pass_off;                         /* -1: plain; else byte offset inside the pass-through pixel */
  int16_t dst_off;                          /* byte offset inside the output pixel (multiple of 16) */
} cdn_pw_chunk;

typedef struct {
  int K;                                    /* input channels actually read: in[p][k_off .. k_off+K) */
  int k_off;                                /* byte offset of the first input channel inside the pixel */
  int N;                                    /* GEMM columns (rows of wq), multiple of 16, <= 1024 */
  int zx;                                   /* zero point of the input QuantAct */
  const int8_t* wq;                         /* host [N][K] integer weights (zero rows/cols for padding) */
  cdn_requant rq;                           /* per GEMM column, n = N */
  const cdn_pw_chunk* chunks; int n_chunks; /* int8 output description (ignored when f32 output is used) */
  /* fp32 NCHW output (head convs): column n < n_f32 goes to d_out_f32[image][n][pixel] with
   * y = acc*Mf[n] + bf[n] (fp64, rounded once to fp32); sigmoid is NOT applied. */
  int n_f32; const double* Mf; const double* bf;
} cdn_pw_desc;

int cdn_pw_gemm_i8(const int8_t* d_in, int in_pitch, int64_t pixels, const cdn_pw_desc* desc,
                   const int8_t* d_pass, int pass_pitch, int8_t* d_out, int out_pitch,
                   float* d_out_f32, int pixels_per_image, cdn_stream_t stream);

/* ---- a whole ShuffleNetV2 unit as ONE kernel ----------------------------------------------------------------
 * QuantBaseNode.forward (portable_quantizer/quant_modules.py:878-907; graph of lib/models/networks/shufflenetv2_dcn.py:57-114):
 *   branch = conv 1x1 (pw1) + BN + ReLU + QuantAct -> depthwise 3x3 (stride 1 | 2) + BN + QuantAct -> conv 1x1 (pw3) + BN + ReLU +
 *   QuantAct;  out = channel_shuffle(cat(pass-through, branch))
 * with the two int8 tensors inside the branch kept in shared memory (DESIGN.md 4.1b).  The three layers are described exactly as for
 * cdn_pw_gemm_i8 / cdn_dw3x3_i8 (pw3 carries the interleaving chunk table); results equal the three separate calls bit for bit.
 *   stride 1: d_x = [B][H][W][2*Hp] in the half layout (pass-through half at byte 0, branch half at byte Hp = pw1->k_off),
 *             d_pass = d_x, Hp = 64 or 128, H % 8 == 0, W % 16 == 0
 *   stride 2: d_x = [B][H][W][32] (24 channels), d_pass = the other branch's output [B][H/2][W/2][pass_pitch], 58 channels per half
 * Returns CDN_ERR_INVALID with cdn_last_error() starting with "unit not fusable" when the shapes / constants are outside what the
 * fused kernels take (wider halves, maps that are not a whole number of 8 x 16 tiles, layers without an exact shift-free
 * requantisation): the caller then issues the three calls. */
int cdn_shuffle_unit_i8(const int8_t* d_x, int x_pitch, int batch, int H, int W, int stride,
                        const cdn_pw_desc* pw1, const int8_t* dw_wq, int dw_C, int dw_zx, const cdn_requant* dw_rq,
                        const cdn_pw_desc* pw3, const int8_t* d_pass, int pass_pitch,
                        int8_t* d_out, int out_pitch, cdn_stream_t stream);

/* ---- ctdet decode ---------------------------------------------------------------------------------------
 * hm: LOGITS fp32 [batch][cat][H][W]; wh, reg: fp32 [batch][2][H][W] (reg may be NULL -> +0.5).
 * Peaks = elements equal to the max of their 3x3 neighbourhood; the K best by (logit desc, class asc, index asc).
 * dets: fp32 [batch][K][6] = x1,y1,x2,y2,sigmoid(logit),class.  inds (optional): int32 [batch][K] = class*H*W+index.
 * If an image has fewer than K peaks the remaining rows are zero and inds = -1. */
int cdn_ctdet_decode(const float* d_hm, const float* d_wh, const float* d_reg, int batch, int cat, int H, int W,
                     int K, float* d_dets, int32_t* d_inds, cdn_stream_t stream);
/* Same with the heat map already holding probabilities (what the reference's ctdet_decode receives after
 * hm.sigmoid_(), lib/detectors/ctdet.py:32): peaks, order and the score written are taken from the values as given. */
int cdn_ctdet_decode_prob(const float* d_heat, const float* d_wh, const float* d_reg, int batch, int cat, int H, int W,
                          int K, float* d_dets, int32_t* d_inds, cdn_stream_t stream);
/* The two calls above allocate their candidate buffer per call and wait for the stream.  The _ws form takes the buffer from
 * the caller (cdn_ctdet_decode_ws_bytes bytes, 8-byte aligned), only enqueues work on `stream`, and can therefore be captured
 * into a CUDA graph; is_prob selects between the two input conventions.  *_img_stride: distance between two images of that
 * tensor in floats (0 = contiguous), so that the three tensors may be channel slices of one [batch][C][H][W] head tensor. */
size_t cdn_ctdet_decode_ws_bytes(int batch, int cat, int H, int W);
int cdn_ctdet_decode_ws(const float* d_hm, long long hm_img_stride, const float* d_wh, long long wh_img_stride,
                        const float* d_reg, long long reg_img_stride, int batch, int cat, int H, int W,
                        int K, int is_prob, float* d_dets, int32_t* d_inds, void* d_ws, size_t ws_bytes, cdn_stream_t stream);

/* ctdet_post_process's coordinate transform on the device (lib/utils/post_process.py:86-103, transform_preds /
 * affine_transform lib/utils/image.py:14-21,58-61): both corners of every box of dets [batch][K][6] (in place) go through
 * the image's inverse affine map h_trans [batch][6] (host doubles, row-major 2x3), evaluated as numpy evaluates
 * np.dot(t, [x, y, 1]) in double and rounded once to float.  Synchronises the stream. */
int cdn_ctdet_post_affine(float* d_dets, int batch, int K, const double* h_trans, cdn_stream_t stream);

/* --flip_test merge of CtdetDetector.process (lib/detectors/ctdet.py:35-38): inputs hold `pairs` (image, mirrored image)
 * couples, hm [2*pairs][cat][H][W] (post-sigmoid) and wh [2*pairs][2][H][W]; out[i] = (in[2i] + flip_W(in[2i+1])) / 2 in fp32,
 * exactly the reference's expression.  reg is taken from the unflipped image by the caller (ctdet.py:38).  Asynchronous. */
int cdn_ctdet_flip_merge(const float* d_hm, const float* d_wh, int pairs, int cat, int H, int W, float* d_out_hm,
                         float* d_out_wh, cdn_stream_t stream);

/* ---- general deformable convolution forward, fp32 (the reference's native plug-in point) ----------------
 * Same argument meaning and order (W before H) as deform_conv_forward_cuda; tensors are contiguous NCHW device
 * pointers: input [B][C][H][W], weight [Co][C/group][kH][kW], offset [B][2*kH*kW*dg][Ho][Wo], output [B][Co][Ho][Wo].
 * im2col_step is accepted and ignored (no im2col buffer exists).  Returns 0 (the reference returns 1). */
int cdn_deform_conv_forward_f32(const float* input, const float* weight, const float* offset, float* output,
                                int B, int C, int H, int W, int Co, int kW, int kH, int dW, int dH,
                                int padW, int padH, int dilW, int dilH, int group, int deformable_group,
                                int im2col_step, cdn_stream_t stream);

/* ---- fused co-designed deformable module, fp32 (the float model's layer) -------------------------------------
 * DeformConvWithOffsetScaleBoundPositive.forward (lib/models/external/modules/dcn_deform_conv.py:323-330) without its
 * optional conv_channel: s = Hardtanh[-bound+1, bound](w_scale . x + b_scale) per output pixel (1x1 conv C -> 1 with
 * stride `stride`), offsets anchor*(s-1), depthwise 3x3 deformable conv (pad 1, bilinear) -- two launches, no offset
 * tensor.  input [B][C][H][W], w_scale [C], w_dw [C][3][3], output [B][C][Ho][Wo] (contiguous NCHW device pointers). */
int cdn_deform_dw_f32(const float* input, const float* w_scale, float b_scale, int offset_bound, const float* w_dw,
                      float* output, int B, int C, int H, int W, int stride, cdn_stream_t stream);
/* cdn_deform_dw_f32 keeps its scratch (the scale scalar per output pixel) in a per-device buffer grown on demand; the _ws
 * form takes it from the caller (cdn_deform_dw_f32_ws_bytes bytes, 8-byte aligned) and never allocates, so it can be captured
 * into a CUDA graph from the first call. */
size_t cdn_deform_dw_f32_ws_bytes(int B, int H, int W, int stride);
int cdn_deform_dw_f32_ws(const float* input, const float* w_scale, float b_scale, int offset_bound, const float* w_dw,
                         float* output, int B, int C, int H, int W, int stride, void* d_ws, size_t ws_bytes, cdn_stream_t stream);
/* The module (stride 1) applied to the nearest x2 upsampling of input [B][C][h][w] without materialising it (the up path's
 * Upsample -> deformable module, lib/models/networks/shufflenetv2_dcn.py:286-300): output [B][C][2h][2w]; workspace
 * cdn_deform_dw_f32_ws_bytes(B, 2h, 2w, 1).  Identical results to upsampling first. */
int cdn_deform_dw_up2_f32_ws(const float* input, const float* w_scale, float b_scale, int offset_bound, const float* w_dw,
                             float* output, int B, int C, int h, int w, void* d_ws, size_t ws_bytes, cdn_stream_t stream);
/* fp32 1x1 convolution NCHW (the module's conv_channel): output [B][Co][P] = weight [Co][C] x input [B][C][P] (+ bias). */
int cdn_pw_f32(const float* input, const float* weight, const float* bias, float* output, int B, int C, int Co,
               int pixels_per_image, cdn_stream_t stream);

/* ---- fp32 NCHW building blocks of the float model (BN folded on the host: conv + bias [+ ReLU]) -------------------
 * Contiguous NCHW device pointers.  cdn_pw_slice_f32 reads input channels [in_coff, in_coff + C) of a tensor with
 * in_ctotal channels and writes output channel out_coff + co*out_cstride of a tensor with out_ctotal channels, which folds
 * split / cat / channel_shuffle (lib/models/networks/shufflenetv2_dcn.py:29-34,102-114) into the indexing;
 * cdn_copy_channels_f32 moves the pass-through half with the same map. */
int cdn_conv3x3_f32(const float* input, const float* weight, const float* bias, float* output, int B, int Ci, int Co,
                    int H, int W, int stride, int relu, cdn_stream_t stream);
int cdn_dw3x3_f32(const float* input, const float* weight, const float* bias, float* output, int B, int C, int H, int W,
                  int stride, int relu, cdn_stream_t stream);
/* The same depthwise conv (stride 1) over the nearest x2 upsampling of `input` [B][C][h][w], which is never materialised:
 * output [B][C][2h][2w].  w must be a multiple of 4. */
int cdn_dw3x3_up2_f32(const float* input, const float* weight, const float* bias, float* output, int B, int C, int h, int w,
                      int relu, cdn_stream_t stream);
int cdn_pw_slice_f32(const float* input, int in_ctotal, int in_coff, int C, const float* weight, const float* bias,
                     float* output, int out_ctotal, int out_coff, int out_cstride, int Co, int relu, int B,
                     int pixels_per_image, cdn_stream_t stream);
/* The same 1x1 convolution on the tensor cores (tcgen05 kind::tf32, csrc/pw_tf32.cu): every product is formed from a 3-way
 * TF32 split (x_hi*w_hi + x_hi*w_lo + x_lo*w_hi, each within ~2^-21 of the exact product); the tensor core only ever sums 16
 * input channels, these chunk sums are added in fp32 (round to nearest) in registers.  The weights are split once:
 * cdn_pw_tf32x3_pack writes the packed array (cdn_pw_tf32x3_packed_floats floats) from the [Co][C] fp32 matrix.
 * pixels_per_image must be a multiple of 256 (CDN_ERR_INVALID otherwise: use cdn_pw_slice_f32); all other arguments as
 * cdn_pw_slice_f32. */
size_t cdn_pw_tf32x3_packed_floats(int Co, int C);
int cdn_pw_tf32x3_pack(const float* d_w, int Co, int C, float* d_packed, cdn_stream_t stream);
int cdn_pw_slice_tf32x3(const float* input, int in_ctotal, int in_coff, int C, const float* d_wpacked,
                        const float* bias, float* output, int out_ctotal, int out_coff, int out_cstride, int Co, int relu,
                        int B, int pixels_per_image, cdn_stream_t stream);
int cdn_copy_channels_f32(const float* input, int in_ctotal, int in_coff, float* output, int out_ctotal, int out_coff,
                          int out_cstride, int n, int B, int pixels_per_image, cdn_stream_t stream);
int cdn_maxpool3s2_f32(const float* input, float* output, int planes, int H, int W, cdn_stream_t stream);
int cdn_upsample2x_f32(const float* input, float* output, int planes, int H, int W, cdn_stream_t stream);

/* ---- whole-network engine -------------------------------------------------------------------------------
 * A plan is a list of tensors (activation buffers) and ops appended in execution order, then finalised for a
 * maximum batch.  All descriptor arrays are copied at add time. */
typedef struct cdn_engine cdn_engine;

int cdn_engine_create(cdn_engine** out, int device);
int cdn_engine_destroy(cdn_engine* e);
/* returns tensor id >= 0; H, W per image; pitch bytes per pixel. */
int cdn_engine_add_tensor(cdn_engine* e, int H, int W, int pitch);
int cdn_engine_add_stem(cdn_engine* e, int out_t, int H, int W, int stride, int pool,
                        const int8_t* wq, int C, const cdn_requant* rq);
int cdn_engine_add_dw(cdn_engine* e, int in_t, int out_t, int in_shift, int stride, const int8_t* wq, int C, int zx,
                      const cdn_requant* rq);
int cdn_engine_add_deform(cdn_engine* e, int in_t, int out_t, int in_shift, const cdn_deform_scale* sc,
                          const int8_t* wq, int C, int zx, const cdn_requant* rq);
/* pass_t = -1 when no chunk interleaves; out_t = -1 for fp32 head output (then f32_slot selects hm/wh/reg via
 * desc->f32 planes: plane index p < cat -> hm[p], cat <= p < cat+2 -> wh, else reg). */
int cdn_engine_add_pw(cdn_engine* e, int in_t, int pass_t, int out_t, const cdn_pw_desc* desc);
int cdn_engine_set_heads(cdn_engine* e, int cat, int H, int W, int K, int has_reg);
int cdn_engine_finalize(cdn_engine* e, int max_batch);
/* d_img: fp32 [batch][3][H][W] on the device.  Outputs (device, may be NULL to skip the copy-out of a map):
 * hm fp32 [batch][cat][Ho][Wo] AFTER sigmoid (ctdet.py:32), wh/reg fp32 [batch][2][Ho][Wo], dets [batch][K][6],
 * inds int32 [batch][K]. */
int cdn_engine_run(cdn_engine* e, const float* d_img, int batch, float* d_hm, float* d_wh, float* d_reg,
                   float* d_dets, int32_t* d_inds, cdn_stream_t stream);
/* Same through HOST buffers: pinned staging, chunked H2D overlapped with compute, D2H of the detections. */
int cdn_engine_run_host(cdn_engine* e, const float* h_img, int batch, float* h_dets, int32_t* h_inds);
/* uint8 input: the image as cv2 hands it to the reference's pre_process (lib/detectors/base_detector.py:48-76),
 * [batch][H][W][3], already at the network's input size.  The normalisation ((u/255. - mean)/std).astype(float32)
 * (:66) is applied inside the stem kernel through a 3x256 table built by cdn_engine_set_normalization with numpy's
 * evaluation order, so results are bit-identical to feeding the normalised fp32 image, at a quarter of the H2D bytes. */
int cdn_engine_set_normalization(cdn_engine* e, const float* mean3, const float* std3);
int cdn_engine_run_u8(cdn_engine* e, const uint8_t* d_img, int batch, float* d_hm, float* d_wh, float* d_reg,
                      float* d_dets, int32_t* d_inds, cdn_stream_t stream);
int cdn_engine_run_host_u8(cdn_engine* e, const uint8_t* h_img, int batch, float* h_dets, int32_t* h_inds);
/* Pipelined host path -- what a prefetching test loop (test.py:62-80: a DataLoader worker prepares image n+1 while the
 * detector runs image n) maps to.  submit enqueues H2D -> forward + decode -> D2H for `slot` (0 or 1) and returns without
 * synchronising; wait blocks until that slot's detections are in h_dets / h_inds.  With both slots in flight the H2D of
 * step n+1 overlaps the compute of step n.  Host buffers must stay valid until wait returns and should be pinned;
 * submitting to a slot that is still in flight is CDN_ERR_STATE. */
int cdn_engine_submit_host(cdn_engine* e, const float* h_img, int batch, float* h_dets, int32_t* h_inds, int slot);
int cdn_engine_submit_host_u8(cdn_engine* e, const uint8_t* h_img, int batch, float* h_dets, int32_t* h_inds, int slot);
int cdn_engine_wait(cdn_engine* e, int slot);
/* Options: "host_chunk" (granularity of the H2D / compute pipeline of run_host: chunks grow x1.6 from host_chunk/2,
 * default 64), "use_graph" (replay the launch sequence as a CUDA graph, default 1), "hm_logits" (cdn_engine_run writes
 * the heat map as logits, what PoseShuffleNetV2.forward returns, instead of post-sigmoid; default 0), "fuse_heads"
 * (default 1: the heads' depthwise conv, QuantDepthwiseNode.forward quant_modules.py:1061-1071, feeds the fp32 output
 * conv inside one kernel, so the int8 tensor between them is not materialised; 0 runs the two plan ops separately,
 * which is what cdn_engine_read_tensor needs to see that tensor.  Same results bit for bit), "fuse_units" (default 1: every
 * eligible stride-1 ShuffleNetV2 unit -- QuantBaseNode.forward, quant_modules.py:878-907: 1x1 conv, depthwise 3x3, 1x1 conv,
 * cat + channel_shuffle -- runs as ONE kernel and the two int8 tensors inside the unit stay on the SM; 2 = the same kernel
 * also writes those two tensors for cdn_engine_read_tensor; 0 = three launches per unit.  The second branch of the first
 * stride-2 unit (1x1 conv at full resolution, depthwise 3x3 stride 2, 1x1 conv + cat + shuffle) is fused the same way.
 * Same results bit for bit). */
int cdn_engine_set_option(cdn_engine* e, const char* name, int value);
/* 1 when the finalized plan runs the heads' tail fused (option on and the layer pair eligible), else 0. */
int cdn_engine_heads_fused(cdn_engine* e);
/* Number of ShuffleNetV2 units of the finalized plan that run as one kernel (option "fuse_units" on and the unit eligible). */
int cdn_engine_units_fused(cdn_engine* e);
/* How plan op i (order of the cdn_engine_add_* calls) runs: 0 = a launch of its own, 1 = first op of the fused heads tail,
 * 2 = first op of a fused stride-1 unit, 3 = first op of the fused branch of the first stride-2 unit, -1 = folded into the
 * launch of an earlier op. */
int cdn_engine_op_fusion(cdn_engine* e, int i);
/* Debug/test access to an activation tensor of the last run: copies batch*H*W*pitch bytes to host. */
int cdn_engine_read_tensor(cdn_engine* e, int tensor, int batch, int8_t* h_out);
/* Raw head outputs of the last run: fp32 [batch][cat+4][Ho*Wo] = hm logits, wh, reg. */
int cdn_engine_read_heads(cdn_engine* e, int batch, float* h_out);
/* Eager run with CUDA events between launches: ms[i] = device time of plan op i, then heads copy-out, then decode
 * (n >= number of ops + 2).  For per-kernel roofline reporting. */
int cdn_engine_profile(cdn_engine* e, const float* d_img, int batch, float* ms, int n, cdn_stream_t stream);
/* Number of kernels one cdn_engine_run launches (for bench.py's gpu_launches). */
int cdn_engine_num_launches(cdn_engine* e);
/* How many int8-producing layers run the exact integer requantisation and how many the guarded fp32 sequence (layers
 * with a channel that has no exact fixed-point form, and the bilinear deformable layers). */
int cdn_engine_requant_stats(cdn_engine* e, int* int_layers, int* guarded_layers);

#ifdef __cplusplus
}
#endif
#endif
