/*
 * esf.h -- C ABI of libesf_b200.so: the sm_100a kernels behind the batched clip forward path of
 * weidafeng/Efficient-SlowFast (`preds = model(inputs)`, SlowFast/tools/test_net.py:92).
 *
 * The reference has no FFI of its own (pure PyTorch: every op below is an ATen -> cuDNN/cuBLAS call in
 * the reference), so each entry point cites the reference nn.Module code it replaces.  The binding a
 * maintainer adds on the reference side is the ctypes stub in INTEGRATION.md; this repo's own binding is
 * efficient_slowfast_b200/runtime.py.
 *
 * Conventions
 *   - plain pointers and sizes only; all pointers are DEVICE pointers unless a name ends in _host;
 *   - activations are channels-last 5-D views (B,T,H,W,C) with element strides (channel stride 1) in one
 *     16-bit storage format per plan -- BF16 or FP16 (view.dtype; all views of a call must agree; tensor-core
 *     operands and packed weights use the same format, accumulation is always FP32); a view may be a channel
 *     slice of a wider concat buffer (C < sW);
 *   - `stream` is a cudaStream_t passed as void*; kernels are enqueued, never synchronised;
 *   - every function returns 0 on success or a negative code; esf_last_error() gives the message of the
 *     last failure on the calling thread; nothing throws, nothing allocates device memory;
 *   - no CPU fallback exists: on a machine without an sm_100 GPU every launch returns an error.
 */
#ifndef ESF_H_
#define ESF_H_
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ESF_OK 0
#define ESF_ERR_ARG (-1)
#define ESF_ERR_CUDA (-2)
#define ESF_ERR_UNSUPPORTED (-3)

#define ESF_ACT_NONE 0
#define ESF_ACT_RELU 1
#define ESF_ACT_RELU6 2

#define ESF_BF16 0
#define ESF_F32 1
#define ESF_F16 2

typedef struct esf_view {
  void* ptr;
  int32_t B, T, H, W, C;
  int64_t sB, sT, sH, sW; /* element strides; channel stride == 1 */
  int32_t dtype;          /* ESF_BF16 / ESF_F16 (16-bit activation storage) or ESF_F32 */
} esf_view;

typedef struct esf_conv_desc {
  esf_view x;           /* BF16 input */
  esf_view y;           /* output, BF16 or F32 (out_dtype) */
  esf_view res;         /* optional BF16 residual added before the activation; ptr == NULL: none */
  const void* w;        /* weights, layout depends on the entry point */
  const float* bias;    /* folded BatchNorm shift (+ conv bias), FP32 */
  int32_t kT, kH, kW;   /* kernel */
  int32_t sT, sH, sW;   /* stride */
  int32_t pT, pH, pW;   /* zero padding */
  int32_t dT, dH, dW;   /* dilation */
  int32_t groups;
  int32_t act;          /* ESF_ACT_* */
  int32_t out_dtype;    /* ESF_BF16 / ESF_F32 */
} esf_conv_desc;

typedef struct esf_op esf_op; /* opaque: one planned kernel launch (TMA descriptors + parameters) */

const char* esf_last_error(void);
int esf_version(void);
/* number of kernel launches issued through this library since load (bench.py's gpu_launches) */
int64_t esf_launch_count(void);

/* ---- dense Conv3d (+ folded BN, + residual, + ReLU) as a tcgen05/TMEM implicit GEMM fed by TMA --------
 * replaces nn.Conv3d + BatchNorm3d(eval) + ReLU (+ residual add) of
 *   BottleneckTransform.forward   SlowFast/slowfast/models/resnet_helper.py:225-240
 *   ResBlock.forward              SlowFast/slowfast/models/resnet_helper.py:352-358
 *   FuseFastToSlow.forward        SlowFast/slowfast/models/video_model_builder.py:143-150
 *   FuseFastAndSlow 1x1x1 convs   SlowFast/slowfast/models/custom_video_model_builder.py:141 and
 *                                 wdf_attention_helper.py:42-48 (query/key/value convs)
 * Weight packing: BF16 [n_pad][taps * kchunks * kc], tap-major then input channel, zero padded; the
 * geometry (kc, kchunks, n_tile, n_pad) for a (cin, cout) pair comes from esf_igemm_geometry(). */
int esf_igemm_geometry(int32_t cin, int32_t cout, int32_t* kc, int32_t* kchunks, int32_t* n_tile, int32_t* n_pad);
int esf_conv_igemm_create(const esf_conv_desc* d, esf_op** out);
/* Same convolution for thin layers (C_in <= 32): a block of WB output columns is folded into the GEMM's N and the
 * input columns it reads into K (banded weights), so TMA rows are 128 B and N = WB * Cout.  Weights: 16-bit band
 * matrix [n_pad][kT*kH*kchunks*64] and tiled bias (engine.pack_wfold_band).  x must be dense in (W, C). */
int esf_conv_wfold_create(const esf_conv_desc* d, int32_t WB, esf_op** out);
int esf_op_launch(esf_op* op, void* stream);
void esf_op_destroy(esf_op* op);

/* ---- direct (CUDA-core) Conv3d for thin layers: grouped / depthwise / Cin < 16 -------------------------
 * replaces the depthwise 3x3x3 / 1xkxk and small pointwise convs of shufflenetv2_helper.py:62-89,
 * shufflenet_helper.py:50-62, mobilenetv2_helper.py:40-55, ghostnet_helper.py:88-143.
 * Weights: FP32 [Cout][kT][kH][kW][Cin/groups]. */
int esf_conv_direct(const esf_conv_desc* d, void* stream);
/* esf_dwconv_padded: the depthwise case of esf_conv_direct for activations whose rows were padded to c_pad (a multiple
 * of 8) channels by the allocator: runs with 16-byte vectors over c_pad channels (zero weights on the padding), e.g.
 * the C = 18 / 162 / 12 / 36 depthwise layers of the fast pathway of SlowFastMoibleNetV2 (mobilenetv2_helper.py:40-55).
 * The caller vouches that channels [C, c_pad) of x, y and res are padding of the same allocation. */
int esf_dwconv_padded(const esf_conv_desc* d, int32_t c_pad, void* stream);
/* esf_pointwise_padded: esf_conv_direct for a 1x1x1 conv whose OUTPUT rows were padded to y_c_pad (a multiple of 8)
 * channels by the allocator: the tiny-channel kernel (C_in < 8 or C_out < 8 -- the first fast-pathway layers, e.g. the
 * 2 -> 12 / 6 -> 36 / 3 -> 18 expansions of mobilenetv2_helper.py:40-55) stores whole 16-byte groups, zeros in the padding,
 * i.e. full 32-byte sectors.  The caller vouches that channels [C, y_c_pad) of y are padding of the same allocation. */
int esf_pointwise_padded(const esf_conv_desc* d, int32_t y_c_pad, void* stream);

/* ---- stem: Conv3d on the FP32 NCDHW clip + folded BN + ReLU -> BF16 channels-last ----------------------
 * replaces ResNetBasicStem.conv/bn/relu (stem_helper.py:173-177) and the efficient stems
 * (stem_helper.py:182-336).  x: FP32 (B,Cin,T,H,W) contiguous.  Weights FP32 [kT][kH][kW][Cin][Cout]. */
int esf_stem_conv(const float* x, int32_t B, int32_t Cin, int32_t T, int32_t H, int32_t W, const float* w,
                  const float* bias, int32_t Cout, int32_t kT, int32_t kH, int32_t kW, int32_t sT, int32_t sH,
                  int32_t sW, int32_t pT, int32_t pH, int32_t pW, int32_t act, const esf_view* y, void* stream);

/* ---- stem on the tensor cores: the Cin = 3 conv as a banded implicit GEMM ---------------------------------
 * Same reference ops as esf_stem_conv (which stays as the generic CUDA-core path for stems whose window does not
 * fit, e.g. very wide kernels).  esf_stem_pack converts the FP32 NCDHW clip to BF16 channels-last rows of `pitch`
 * elements with explicit left/right zero padding; esf_stem_igemm_create plans the GEMM (launch with
 * esf_op_launch).  w_band: BF16 [n_pad][kT*kH*64] band matrix, bias_tiled: FP32 [n_pad] (layout documented in
 * csrc/esf_igemm.cu and built by engine.pack_stem_band). Temporal stride must be 1. */
int esf_stem_geometry(int32_t W, int32_t Cin, int32_t kW, int32_t sW, int32_t pW, int32_t* pitch, int32_t* lpad,
                      int32_t* window);
int esf_stem_pack(const float* x, int32_t B, int32_t Cin, int32_t T, int32_t H, int32_t W, int32_t pitch,
                  int32_t lpad, int32_t dtype, void* xp, void* stream);
/* esf_stem_pack_gather: esf_stem_pack of the SLOW pathway straight out of the FAST pathway's clip.  The loader's
 * pack_pathway_output (SlowFast/slowfast/datasets/utils.py:93-102) makes slow = fast[:, :, linspace(0, T-1, T/alpha)]:
 * the same pixels twice.  x: FP32 (B, Cin, Tsrc, H, W) fast clip; t_index: device int32[T], source frame of every slow
 * frame -- the slow clip is never uploaded nor materialised (ClipStream(slow_from_fast=True)). */
int esf_stem_pack_gather(const float* x, int32_t B, int32_t Cin, int32_t Tsrc, int32_t H, int32_t W,
                         const int32_t* t_index, int32_t T, int32_t pitch, int32_t lpad, int32_t dtype, void* xp,
                         void* stream);
/* ---- uint8 frame input (SURVEY 8-f4) ---------------------------------------------------------------------
 * Replaces the loader-side chain the reference runs on the host before the H2D copy: tensor_normalize
 * (SlowFast/slowfast/datasets/utils.py:298-315: u8 -> float / 255, - mean, / std), permute(3,0,1,2)
 * (datasets/kinetics.py:231-235) and pack_pathway_output (datasets/utils.py:73-112: channel reversal, slow-pathway
 * frame gather by index).  frames: device uint8 (B, Tsrc, H, W, C) contiguous, C <= 4.  t_index: device int32[T]
 * source frame of every output frame, or null for the identity (then T == Tsrc).  chan_src: host int32[C], source
 * channel of every output channel, or null for the identity.  The look-up tables are built by the caller with the
 * reference's own FP32 operations: lut[c * 256 + u] = normalised value of byte u in output channel c.
 * esf_stem_pack_u8 writes the packed stem rows of esf_stem_pack directly (lut16: 16-bit values in the plan's
 * storage format); esf_frames_to_clip writes the FP32 (B, C, T, H, W) clip for stems that read NCDHW (lut32). */
int esf_stem_pack_u8(const uint8_t* frames, int32_t B, int32_t Tsrc, int32_t H, int32_t W, int32_t C,
                     const int32_t* t_index, int32_t T, const int32_t* chan_src, const void* lut16, int32_t pitch,
                     int32_t lpad, void* xp, void* stream);
int esf_frames_to_clip(const uint8_t* frames, int32_t B, int32_t Tsrc, int32_t H, int32_t W, int32_t C,
                       const int32_t* t_index, int32_t T, const int32_t* chan_src, const float* lut32, float* clip,
                       void* stream);
/* The same two outputs gathered from a bank of per-camera frame rings (the demo loop over many cameras,
 * efficient_slowfast_b200/demo.py CameraWindows): bank: device uint8 (N, L, H, W, C) contiguous, camera n's ring of its
 * last L frames.  rows: device int32[R][2], (camera, oldest ring slot) of every output row.  pos: device int32[T], the
 * pathway's window positions (oldest frame = 0, demo.window_indices).  Output row r, frame t is ring slot
 * (pos[t] + oldest_r) % L of camera camera_r, so a call uploads only the 8 * R bytes of rows.  rows_host / pos_host:
 * the same tables on the host, read for the range checks before the launch: R >= 1, camera in [0, N), oldest and pos
 * entries in [0, L).  chan_src, tables and outputs as esf_stem_pack_u8 / esf_frames_to_clip with B = R rows. */
int esf_stem_pack_u8_rings(const uint8_t* bank, int32_t N, int32_t L, int32_t H, int32_t W, int32_t C,
                           const int32_t* rows, const int32_t* rows_host, int32_t R, const int32_t* pos,
                           const int32_t* pos_host, int32_t T, const int32_t* chan_src, const void* lut16, int32_t pitch,
                           int32_t lpad, void* xp, void* stream);
int esf_frames_to_clip_rings(const uint8_t* bank, int32_t N, int32_t L, int32_t H, int32_t W, int32_t C,
                             const int32_t* rows, const int32_t* rows_host, int32_t R, const int32_t* pos,
                             const int32_t* pos_host, int32_t T, const int32_t* chan_src, const float* lut32,
                             float* clip, void* stream);
/* ---- test-time spatial sampling of uint8 frames (csrc/esf_crop.cu) -------------------------------------------------
 * The same chain with the reference's test-mode spatial_sampling in between (SlowFast/slowfast/datasets/utils.py
 * spatial_sampling -> transform.random_short_side_scale_jitter with min = max = crop size S, bilinear
 * F.interpolate(align_corners=False), then transform.uniform_crop at spatial_idx 0/1/2), from frames at decode size
 * (B, Tsrc, H0, W0, C).  Output row b * V + v is source clip b cropped at view v.  The resize to Hr x Wr is given as
 * per-axis tables built on the host (efficient_slowfast_b200/frames.py axis_table): y_index[2 * r + k] / y_weight[2 * r + k]
 * are the source rows i0, i1 and weights l0, l1 of resized row r (x_* the same for columns); they may be null when
 * Hr == H0 and Wr == W0 (a pure window).  crop_yx_host: host int32[2 * V], (y0, x0) of every view in the resized frame,
 * V <= 8; each crop must lie inside it.  W0 * C <= 16384.  lut32 as esf_frames_to_clip.
 * esf_stem_pack_u8_crop writes the packed stem rows of esf_stem_pack ([B * V][T][S][pitch], dtype ESF_BF16 / ESF_F16);
 * esf_frames_to_clip_crop the FP32 (B * V, C, T, S, S) clip. */
int esf_stem_pack_u8_crop(const uint8_t* frames, int32_t B, int32_t Tsrc, int32_t H0, int32_t W0, int32_t C,
                          const int32_t* t_index, int32_t T, const int32_t* chan_src, const float* lut32,
                          const int32_t* y_index, const float* y_weight, int32_t Hr, const int32_t* x_index,
                          const float* x_weight, int32_t Wr, const int32_t* crop_yx_host, int32_t V, int32_t S,
                          int32_t dtype, int32_t pitch, int32_t lpad, void* xp, void* stream);
int esf_frames_to_clip_crop(const uint8_t* frames, int32_t B, int32_t Tsrc, int32_t H0, int32_t W0, int32_t C,
                            const int32_t* t_index, int32_t T, const int32_t* chan_src, const float* lut32,
                            const int32_t* y_index, const float* y_weight, int32_t Hr, const int32_t* x_index,
                            const float* x_weight, int32_t Wr, const int32_t* crop_yx_host, int32_t V, int32_t S,
                            float* clip, void* stream);
/* The same for a batch of B clips of mixed decode sizes (one Tsrc, C for all): clip b is (Tsrc, H0_b, W0_b, C) uint8 at
 * the device address frames_host[b] (a host array of B addresses).  geom_host: host int32[B][4], (H0, W0, Hr, Wr) of
 * every clip; tables_host: host array [B][4] of the device addresses of its y_index, y_weight, x_index, x_weight (null
 * allowed where the clip is not resized); crop_yx_host: host int32[B][V][2].  Output row b * V + v is clip b at view v,
 * as above.  Every clip is checked before anything is launched; the host arrays are read before the call returns. */
int esf_stem_pack_u8_crop_ragged(const void* frames_host, int32_t B, int32_t Tsrc, int32_t C, const int32_t* t_index,
                                 int32_t T, const int32_t* chan_src, const float* lut32, const int32_t* geom_host,
                                 const void* tables_host, const int32_t* crop_yx_host, int32_t V, int32_t S,
                                 int32_t dtype, int32_t pitch, int32_t lpad, void* xp, void* stream);
int esf_frames_to_clip_crop_ragged(const void* frames_host, int32_t B, int32_t Tsrc, int32_t C, const int32_t* t_index,
                                   int32_t T, const int32_t* chan_src, const float* lut32, const int32_t* geom_host,
                                   const void* tables_host, const int32_t* crop_yx_host, int32_t V, int32_t S,
                                   float* clip, void* stream);
/* Temporal views of whole videos (the reference's test loader: NUM_ENSEMBLE_VIEWS temporal clips per video, each then
 * resized and cropped as above).  Clip b is one (video, temporal view) pair: frames_host[b] is the device address of
 * its video (Tsrc_b, H0_b, W0_b, C) uint8, and views of one video share that address.  geom_host: host int32[B][5],
 * (Tsrc, H0, W0, Hr, Wr) of every clip; t_index: DEVICE int32[B][T], row b the source frames of clip b (required;
 * every entry is clamped to [0, Tsrc_b - 1]); tables_host and crop_yx_host as for the ragged entry points.  Output row
 * b * V + v is clip b at view v.  Every clip is checked before anything is launched; the host arrays are read before
 * the call returns. */
int esf_stem_pack_u8_crop_videos(const void* frames_host, int32_t B, int32_t C, const int32_t* t_index, int32_t T,
                                 const int32_t* chan_src, const float* lut32, const int32_t* geom_host,
                                 const void* tables_host, const int32_t* crop_yx_host, int32_t V, int32_t S,
                                 int32_t dtype, int32_t pitch, int32_t lpad, void* xp, void* stream);
int esf_frames_to_clip_crop_videos(const void* frames_host, int32_t B, int32_t C, const int32_t* t_index, int32_t T,
                                   const int32_t* chan_src, const float* lut32, const int32_t* geom_host,
                                   const void* tables_host, const int32_t* crop_yx_host, int32_t V, int32_t S,
                                   float* clip, void* stream);
/* ---- AVA detection from uint8 frames (csrc/esf_crop.cu) ----------------------------------------------------------------
 * The test split of the reference's AVA loader (SlowFast/slowfast/datasets/ava_dataset.py _images_and_boxes_preprocessing,
 * PyTorch backend): u / 255 -> short-side bilinear resize to Hr x Wr (transform.random_short_side_scale_jitter, no
 * crop) -> color_normalization -> channel swap -> pack_pathway_output, from frames at decode size (B, Tsrc, H0, W0, C).
 * The resize runs on the [0, 1] values and the normalisation after it: lut32 is the [C][256] table of u / 255 (per
 * OUTPUT channel, as esf_frames_to_clip), mean_host / std_host: host float[C], the statistics of every SOURCE channel
 * (output channel c = source channel chan_src[c] takes those of its source).  Resize tables as esf_stem_pack_u8_crop
 * (null when Hr == H0 and Wr == W0).  Output row b is clip b's whole Hr x Wr frame: packed stem rows [B][T][Hr][pitch]
 * (pitch >= lpad + Wr * C) or the FP32 (B, C, T, Hr, Wr) clip. */
int esf_stem_pack_u8_ava(const uint8_t* frames, int32_t B, int32_t Tsrc, int32_t H0, int32_t W0, int32_t C,
                         const int32_t* t_index, int32_t T, const int32_t* chan_src, const float* lut32,
                         const float* mean_host, const float* std_host, const int32_t* y_index, const float* y_weight,
                         int32_t Hr, const int32_t* x_index, const float* x_weight, int32_t Wr, int32_t dtype,
                         int32_t pitch, int32_t lpad, void* xp, void* stream);
int esf_frames_to_clip_ava(const uint8_t* frames, int32_t B, int32_t Tsrc, int32_t H0, int32_t W0, int32_t C,
                           const int32_t* t_index, int32_t T, const int32_t* chan_src, const float* lut32,
                           const float* mean_host, const float* std_host, const int32_t* y_index, const float* y_weight,
                           int32_t Hr, const int32_t* x_index, const float* x_weight, int32_t Wr, float* clip,
                           void* stream);
/* The same branch's boxes: boxes (K, 5) on the device, FP32 (f64 = 0) or FP64 (f64 = 1), rows [batch index, x1, y1, x2,
 * y2] with coordinates in [0, 1] of the H0 x W0 frames; out: FP32 (K, 5) in pixels of the Hr x Wr frames.  FP64 as the
 * loader's numpy: times (W0, H0), clip_boxes_to_image(H0, W0), times new / old of the short-side resize (none when
 * Hr == H0 and Wr == W0), clip_boxes_to_image(S, S) with S the crop size; the batch index is passed through.  No
 * host synchronisation. */
int esf_ava_boxes(const void* boxes, int32_t f64, int32_t K, int32_t H0, int32_t W0, int32_t Hr, int32_t Wr, int32_t S,
                  float* out, void* stream);
/* ---- the demo's frame resize (csrc/esf_crop.cu) -------------------------------------------------------------------------
 * cv2.resize(frame, (Ws, Hs), interpolation=cv2.INTER_LINEAR) on uint8 frames, as the reference demo's
 * datasets/cv2_transform.scale runs it on every captured frame: OpenCV's fixed-point arithmetic (11-bit weights) in
 * integers, bit for bit.  One call resizes B frames of their own sizes: frames_host / dst_host are host arrays of B
 * device addresses, frame b being (H, W, C) uint8 contiguous and its output (Hs, Ws, C) uint8 contiguous (a camera's
 * ring slot).  geom_host: host int32[B][4], (H, W, Hs, Ws).  tables_host: host array [B][2] of the device addresses
 * (8-byte aligned) of the y table [Hs] and the x table [Ws], entries {int32 source index; int16 w0; int16 w1} as
 * efficient_slowfast_b200/frames.py cv2_axis_table makes them.  C is 1, 3 or 4 (OpenCV takes another route for the
 * exact 2x downscale of 2-channel frames); W * C <= 16384.  Every frame is checked before anything is launched; the
 * host arrays are read before the call returns. */
int esf_resize_u8_cv2(const void* frames_host, const void* dst_host, const int32_t* geom_host, const void* tables_host,
                      int32_t B, int32_t C, void* stream);
/* ---- baseline JPEG decoding (csrc/esf_jpeg.cu) --------------------------------------------------------------------------
 * cv2.imdecode(buf, cv2.IMREAD_COLOR) (BGR) or, with gray, cv2.IMREAD_GRAYSCALE, bit for bit (OpenCV's libjpeg-turbo with
 * its defaults: islow IDCT, fancy upsampling), for the frame-directory loaders' cv2.imread.  Baseline / extended
 * sequential Huffman files of 8-bit precision, one interleaved scan, 1 component or 3 YCbCr components with luma
 * sampling 1x1, 2x1, 2x2, 1x2 or 4x1 and 1x1 chroma.  efficient_slowfast_b200/jpeg.py parses the files and packs `blob`
 * (device, 16-byte aligned, blob_bytes long), sections 16-byte aligned in this order:
 *   esf_jpeg_file[n_files], esf_jpeg_segment[n_segs], n_huff Huffman tables of 1424 bytes (uint16 look[512]: code
 *   length << 8 | symbol of the 9-bit codes' prefixes, 0 for longer codes; int32 maxcode[18]; int32 valoffset[18];
 *   uint8 values[256], as libjpeg's jpeg_make_d_derived_tbl), n_quant quantisation tables (int16[64], natural order),
 *   then the files' bytes, which segment offsets count from.
 * files_host / segs_host are host copies of the first two sections; every descriptor is checked on them before anything
 * is launched.  Segments are grouped by file in file order, one per restart interval (first_mcu = k * restart) or one per
 * scan.  scratch: esf_jpeg_scratch_bytes bytes (16-byte aligned).  out: (n_files, H, W, C) uint8 contiguous, C = 3 or
 * C = 1 with gray; every file is H x W.  status: device int32[n_files], zeroed, then nonzero for a file whose scan holds
 * an invalid Huffman code (its pixels are then unspecified; nothing is written outside its frame). */
typedef struct esf_jpeg_file {
  int32_t H, W, ncomp, restart; /* restart interval in MCUs, 0: the scan is one segment */
  int32_t h[3], v[3];           /* sampling factors (1, 1 for a one-component file) */
  int32_t qt[3], dc[3], ac[3];  /* per component: quantisation and Huffman table indices into the blob's sections */
  int32_t pad;
} esf_jpeg_file;
typedef struct esf_jpeg_segment {
  int64_t begin, end;           /* entropy-coded bytes, markers and fill bytes excluded */
  int32_t file, first_mcu;
} esf_jpeg_segment;
int esf_jpeg_scratch_bytes(const esf_jpeg_file* files_host, int32_t n_files, int32_t gray, int64_t* bytes);
int esf_jpeg_decode(const void* blob, int64_t blob_bytes, const esf_jpeg_file* files_host, int32_t n_files,
                    const esf_jpeg_segment* segs_host, int32_t n_segs, int32_t n_huff, int32_t n_quant, void* scratch,
                    int64_t scratch_bytes, uint8_t* out, int32_t H, int32_t W, int32_t C, int32_t gray, void* status,
                    void* stream);
int esf_stem_igemm_create(const void* xp, int32_t B, int32_t Cin, int32_t T, int32_t H, int32_t W, int32_t pitch,
                          const void* w_band, const float* bias_tiled, int32_t Cout, int32_t kT, int32_t kH,
                          int32_t kW, int32_t sH, int32_t sW, int32_t pT, int32_t pH, int32_t pW, int32_t act,
                          const esf_view* y, esf_op** out);
/* Temporal-band stem for kT > 1 (the fast pathway's 5x7x7 stem, stem_helper.py:138-178 with cfg.SLOWFAST.BETA_INV):
 * same operands and packed clip as esf_stem_igemm_create, but the kT time taps are folded into the GEMM's N and the
 * input frames stream past an M tile that stays on its SM (output frames accumulate in a ring of TMEM slots).
 * esf_stem_tband_wb: width WB of the output-column block for this geometry, 0 when the kernel does not apply (kT = 1,
 * window or N too large).  w_band: 16-bit [kT*WB*Cout][kH*64], bias_tiled: FP32 [WB*Cout] (engine.pack_stem_tband).
 * Dense output, 16-bit or FP32 (raw accumulators of a split product of the FP32-accurate plan). */
int esf_stem_tband_wb(int32_t W, int32_t Cin, int32_t Cout, int32_t kT, int32_t kH, int32_t kW, int32_t sW, int32_t pW);
int esf_stem_tband_create(const void* xp, int32_t B, int32_t Cin, int32_t T, int32_t H, int32_t W, int32_t pitch,
                          const void* w_band, const float* bias_tiled, int32_t Cout, int32_t kT, int32_t kH,
                          int32_t kW, int32_t sH, int32_t sW, int32_t pT, int32_t pH, int32_t pW, int32_t act,
                          const esf_view* y, esf_op** out);

/* ---- MaxPool3d / AvgPool3d on channels-last BF16 (padding: -inf for max, zeros counted for avg) ---------
 * replaces ResNetBasicStem.pool_layer (stem_helper.py:169-171), the 3x3x3 stem pools
 * (stem_helper.py:243,281) and the ShuffleNet shortcut AvgPool3d (shufflenet_helper.py:68-73). */
int esf_pool3d(const esf_view* x, const esf_view* y, int32_t kT, int32_t kH, int32_t kW, int32_t sT, int32_t sH,
               int32_t sW, int32_t pT, int32_t pH, int32_t pW, int32_t is_avg, int32_t act, void* stream);

/* ---- channel plumbing of the efficient backbones (BF16 views, any channel count) ---------------------------
 * esf_shuffle_concat: y = channel_shuffle(cat(a, b), groups)   (shufflenetv2_helper.py:32-43,104-112,
 *                     shufflenet_helper.py:24-34,77); b may be NULL.
 * esf_eltwise_add:    y = act(a + b)                           (ghostnet_helper.py:161-162 residual add)
 * esf_channel_scale:  y = x * scale[b][c]                      (SqueezeExcite gate, ghostnet_helper.py:46-52) */
int esf_shuffle_concat(const esf_view* a, const esf_view* b, int32_t groups, const esf_view* y, void* stream);
int esf_eltwise_add(const esf_view* a, const esf_view* b, const esf_view* y, int32_t act, void* stream);
int esf_channel_scale(const esf_view* x, const float* scale, const esf_view* y, void* stream);

/* ---- CMDA fast->slow: MaxPool(alpha,1,1) -> ECA -> BN -> ReLU -> write into the slow concat slice ------
 * replaces FuseFastAndSlow.forward lines custom_video_model_builder.py:131-135 and ECA.forward
 * (wdf_attention_helper.py:77-91).  Two launches: (1) per-(clip,channel) partial sums of the temporally
 * max-pooled tensor, (2) channel conv1d + sigmoid + scale + BN affine + ReLU + store.
 * partial: FP32 scratch of esf_eca_scratch_floats(B, C) elements. */
int64_t esf_eca_scratch_floats(int32_t B, int32_t C);
int esf_eca_fuse(const esf_view* x_fast, int32_t alpha, const float* eca_w, int32_t eca_k, const float* bn_scale,
                 const float* bn_shift, float* partial, const esf_view* y_slow_slice, void* stream);

/* ---- CMDA slow->fast position attention, fused (never materialises the N x N affinity) ------------------
 * replaces SpatialAttention.forward (wdf_attention_helper.py:33-54) + bn_s2f + ReLU + nearest upsample +
 * concat (custom_video_model_builder.py:142-146).
 *   proj: FP32 (B*N, 4*d) rows [x_d | q | k | v] produced by the composed 1x1x1 GEMM (out_dtype F32);
 *   y[b, alpha*t + r, h, w, 0:d] = relu(bn_scale * (gamma * O + x_d) + bn_shift), r = 0..alpha-1, where
 *   O = softmax_j(q_i.k_j) v_j runs on the tcgen05 tensor cores (TMEM accumulators, two-pass softmax), any head dim
 *   d <= 128.  esf_attn_tc_pack writes Q~/K~ (hi/lo split rows, so QK^T keeps ~FP32 logits on 16-bit tensor cores),
 *   V^T and x_d into `packed` (esf_attn_tc_pack_bytes bytes); esf_attn_tc_create plans the fused kernel (launch:
 *   esf_op_launch). */
int64_t esf_attn_tc_pack_bytes(int32_t B, int32_t N, int32_t d);
int esf_attn_tc_pack(const float* proj, int32_t B, int32_t N, int32_t d, int32_t dtype, void* packed, void* stream);
int esf_attn_tc_create(const void* packed, int32_t B, int32_t T, int32_t H, int32_t W, int32_t d, float gamma,
                       const float* bn_scale, const float* bn_shift, int32_t alpha, const esf_view* y_fast_slice,
                       esf_op** out);

/* (esf_attn_tc_create also accepts an FP32 output view: the FP32-accurate path below; operands are then FP16.) */

/* ---- generic CUDA-core fallback of the same attention for head dims the tensor-core kernels do not cover (d > 128;
 * in the reference's models that only happens with N <= 392 keys).  Reads the FP32 projection rows directly; the
 * output view is BF16, F16 or F32 (FP32 math throughout: the FP32-accurate plan uses it above d = 128 too). */
int esf_attn_generic(const float* proj, int32_t B, int32_t T, int32_t H, int32_t W, int32_t d, float gamma,
                     const float* bn_scale, const float* bn_shift, int32_t alpha, const esf_view* y_fast_slice,
                     void* stream);

/* ---- Non-local block glue (SURVEY 8-f3; SlowFast/slowfast/models/nonlocal_helper.py:105-148) ------------------
 * The block's two matrix products (theta^T phi and (.) g^T, einsum lines 122 / 139) are launched per clip as
 * esf_conv_igemm_create GEMMs whose weight matrix is the clip's own phi rows / transposed g rows; the 1x1x1 convs
 * theta / phi / g / out, the max-pool and the residual + BN are the ordinary conv / pool entry points.
 * esf_row_softmax normalises the FP32 affinity rows S[rows][n] (pitch s_pitch) into 16-bit P (pitch p_pitch):
 *   mode 0: softmax_j(scale * S) ("softmax", scale = dim_inner^-0.5);  mode 1: scale * S ("dot_product", 1 / n).
 * esf_transpose16: out[b][c][r] = in[b][r][c] on 16-bit elements (g rows -> g^T, the GEMM's [n][k] weight layout). */
/* esf_gemm_clip_weights_create: the 1x1x1 implicit GEMM of esf_conv_igemm_create with one weight matrix PER CLIP --
 * d->w points at B stacked matrices ([B][n_pad][kchunks * kc] 16-bit), d->bias at one shared FP32 [n_pad] vector; an
 * M tile never spans two clips.  One launch computes theta^T phi (or P g^T) of every clip of the batch. */
int esf_gemm_clip_weights_create(const esf_conv_desc* d, esf_op** out);
int esf_row_softmax(const float* S, int64_t rows, int32_t n, int64_t s_pitch, float scale, int32_t mode, int32_t dtype,
                    void* P, int64_t p_pitch, void* stream);
int esf_transpose16(const void* in, int32_t B, int32_t rows, int32_t cols, int64_t in_bstride, int64_t in_pitch, void* out,
                    int64_t out_bstride, int64_t out_pitch, void* stream);

/* ---- head: global average pool of each pathway -> concat -> Linear -> softmax/ReLU/none -----------------
 * replaces ResNetBasicHead.forward eval branch (head_helper.py:198-223) and the efficient heads'
 * pool+classifier tails.  feat: FP32 scratch (B, C0 + C1).  act: 0 none (logits), 1 softmax, 2 relu, 3 sigmoid,
 * 4 hard-sigmoid (the same kernel serves the squeeze-excite MLP of ghostnet_helper.py:46-52). */
int esf_head_pool(const esf_view* x0, const esf_view* x1, float* feat, void* stream);
int esf_head_fc(const float* feat, int32_t B, int32_t Cin, int32_t feat_stride, const float* w, const float* bias,
                int32_t num_classes, int32_t act, float* out, int32_t out_stride, void* stream);
/* esf_global_mean: the same global average as esf_head_pool for LARGE activations (the squeeze of SqueezeExcite,
 * ghostnet_helper.py:46-52, sees up to 32 x 56 x 56 positions): 64 deterministic partial sums per clip in `scratch`
 * (esf_global_mean_scratch_floats(B, C) floats), then their sum.  feat[b][feat_off + c] = mean_{t,h,w} x[b,t,h,w,c]. */
int64_t esf_global_mean_scratch_floats(int32_t B, int32_t C);
int esf_global_mean(const esf_view* x, float* scratch, float* feat, int32_t feat_stride, int32_t feat_off, void* stream);
/* Fully-convolutional inference (head_helper.py:218-220: `x = self.act(x); x = x.mean([1, 2, 3])`) when the head's
 * AvgPool3d kernel is smaller than the feature map (e.g. TEST_CROP_SIZE 256 on a 224 model): esf_pool3d (avg, stride
 * 1) -> esf_head_pool / esf_head_fc with one row per (clip, position) -> esf_group_mean over the P positions:
 * out[b][k] = mean_p in[b][p][k]. */
int esf_group_mean(const float* in, int32_t B, int32_t P, int32_t K, float* out, void* stream);

/* ---- RoI head of the AVA detection models (ResNetRoIHead, head_helper.py:12-130; csrc/esf_roi.cu) ----------------
 * esf_temporal_mean: y[b][h][w][c] = mean_t x[b, t, h, w, c] -- the head's AvgPool3d([T, 1, 1]) when it leaves one
 *   frame; x: 16-bit view, y: dense FP32 (B, H, W, C).
 * esf_roi_align_max: feat[k][c_off + c] = max over the R x R bins of RoIAlign(R, spatial_scale, sampling_ratio 0,
 *   aligned) on map[b_k] (torchvision roi_align semantics, as detectron2's ROIAlign), i.e. RoIAlign + MaxPool2d(R).
 *   map: dense FP32 (B, H, W, C); boxes: FP32 (K, 5) rows [batch index, x1, y1, x2, y2] in input pixels.  The batch
 *   index is clamped to [0, B); a box with non-finite geometry gives a NaN row; the adaptive sampling grid of a bin is
 *   capped at 64 x 64.  One row per box, deterministic (no atomics); both pathways write slices of one row. */
int esf_temporal_mean(const esf_view* x, float* y, void* stream);
int esf_roi_align_max(const float* map, int32_t B, int32_t H, int32_t W, int32_t C, const float* boxes, int32_t K,
                      float spatial_scale, int32_t resolution, int32_t aligned, float* feat, int32_t feat_stride,
                      int32_t c_off, void* stream);

/* ---- FP32-accurate path (cfg.ESF.PRECISION = "fp32"; north star: rel err <= 1e-4 against the reference's FP32 forward) --
 * The reference is FP32 end to end (resnet_helper.py:182-240, wdf_attention_helper.py:42-53).  Here every tensor-core
 * operand is a pair of FP16 numbers x = hi + lo (22 mantissa bits) and x.w = x_hi.w_hi + x_lo.w_hi + x_hi.w_lo, evaluated
 * by the SAME implicit GEMM (esf_conv_igemm_create, FP32 output): activations are stored as three channel planes
 * [hi | lo | hi] (plane pitch `plane` elements) and the folded weights as [w_hi | w_hi | w_lo] along the input-channel
 * axis, i.e. an ordinary convolution with 3x the input channels.  The entry points below are the FP32 element-wise glue:
 *   esf_p32_post:      v = act(acc * scale[c] + bias[c] + res); y32 = v (optional); y3 = planes of v (optional).
 *                      acc / res / y32: FP32 views; y3: FP16 view of the hi plane's channel slice (lo at + plane,
 *                      second hi at + 2 * plane elements; weight_order = 1: [hi | hi | lo] instead).  scale undoes the
 *                      power-of-two row scaling of the weights.
 *   esf_p32_pool3d:    MaxPool3d / AvgPool3d on FP32 views (stem_helper.py:169-171).
 *   esf_p32_eca_fuse:  the FP32 form of esf_eca_fuse (custom_video_model_builder.py:131-135); partial:
 *                      esf_p32_eca_scratch_floats(B, C) floats; C must divide 256.
 *   esf_p32_head_pool: feat[b][feat_off + c] = mean_{t,h,w} x (head_helper.py:198-210) on an FP32 view.
 *   esf_p32_attention: SpatialAttention.forward (wdf_attention_helper.py:33-54) + bn_s2f + ReLU + x alpha upsample in
 *                      FP32 on the CUDA cores (flash style, no N x N matrix); proj: FP32 rows [x_d | q | k | v];
 *                      any d <= 128.  (The tcgen05 attention rounds P and V to FP16.)
 * esf_stem_conv accepts an FP32 output view (FP32 CUDA-core stem) and esf_attn_tc_create an FP32 output slice. */
int esf_p32_post(const esf_view* acc, const float* scale, const float* bias, const esf_view* res, int32_t act,
                 const esf_view* y32, const esf_view* y3, int32_t plane, int32_t weight_order, void* stream);
/* esf_p32_post3: v = act((acc + acc2 + acc3) * scale + bias) -> y32 / planes: the banded stem GEMM runs its three split
 * products as three launches (esf_stem_igemm_create with an FP32 output view; esf_stem_pack_lo packs the low halves of
 * the clip: xp_lo = fp16(x - fp16(x))). */
int esf_p32_post3(const esf_view* acc, const esf_view* acc2, const esf_view* acc3, const float* scale, const float* bias,
                  int32_t act, const esf_view* y32, const esf_view* y3, int32_t plane, void* stream);
int esf_stem_pack_lo(const float* x, int32_t B, int32_t Cin, int32_t T, int32_t H, int32_t W, int32_t pitch, int32_t lpad,
                     int32_t dtype, void* xp, void* stream);
/* Non-local block in this mode (nonlocal_helper.py:105-148): the clip's own phi / g rows are the "weights" of the two
 * products, so they are stored in weight order [hi | hi | lo] (esf_p32_post weight_order = 1); esf_p32_row_softmax
 * turns the FP32 affinity rows into the [hi | lo | hi] planes of softmax(scale * S) (mode 0) or scale * S (mode 1). */
int esf_p32_row_softmax(const float* S, int64_t rows, int32_t n, int64_t s_pitch, float scale, int32_t mode, void* P3,
                        int64_t p_pitch, int32_t plane, void* stream);
int esf_p32_pool3d(const esf_view* x, const esf_view* y, int32_t kT, int32_t kH, int32_t kW, int32_t sT, int32_t sH,
                   int32_t sW, int32_t pT, int32_t pH, int32_t pW, int32_t is_avg, void* stream);
int64_t esf_p32_eca_scratch_floats(int32_t B, int32_t C);
int esf_p32_eca_fuse(const esf_view* x_fast, int32_t alpha, const float* eca_w, int32_t eca_k, const float* bn_scale,
                     const float* bn_shift, float* partial, const esf_view* y, void* stream);
int esf_p32_head_pool(const esf_view* x, float* feat, int32_t feat_stride, int32_t feat_off, void* stream);
/* The same attention on the tensor cores at FP32 accuracy for d <= 64 ("split mode" of the one-row-per-thread tcgen05
 * kernel): logits are hi/lo split already; here P and V are FP16 PAIRS as well, O += P_hi V_hi + P_lo V_hi + P_hi V_lo,
 * row sums in FP32 registers.  esf_attn_tc_pack (dtype F16) fills `packed`; esf_attn_tc_pack_vlo writes V_lo^T
 * (esf_attn_tc_vlo_bytes bytes, the layout of V^T); esf_attn_tc_create_split plans the launch (FP32 output view). */
int64_t esf_attn_tc_vlo_bytes(int32_t B, int32_t N, int32_t d);
int esf_attn_tc_pack_vlo(const float* proj, int32_t B, int32_t N, int32_t d, void* v_lo, void* stream);
int esf_attn_tc_create_split(const void* packed, const void* v_lo, int32_t B, int32_t T, int32_t H, int32_t W, int32_t d,
                             float gamma, const float* bn_scale, const float* bn_shift, int32_t alpha,
                             const esf_view* y_fast_slice, esf_op** out);
int esf_p32_attention(const float* proj, int32_t B, int32_t T, int32_t H, int32_t W, int32_t d, float gamma,
                      const float* bn_scale, const float* bn_shift, int32_t alpha, const esf_view* y, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* ESF_H_ */
