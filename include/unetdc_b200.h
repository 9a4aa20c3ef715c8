/*
 * unetdc_b200.h -- C ABI of libunetdc_b200.so: the B200 (sm_100a) implementation of the
 * inference + quantification hot path behind the reference's quantify_droplets_batch.py.
 *
 * The reference (malani86/unet-DC-segmentation) is pure Python and has no FFI; the boundary
 * it offers is the Python call surface quantify_droplets_batch.py itself uses (SURVEY.md 8b).
 * Each entry point below replaces the device work of one of those calls; the Python mirror in
 * unet_dc_segmentation_b200/ binds them with ctypes (see INTEGRATION.md):
 *
 *   dc_model_* / dc_forward      UNetDC.__call__            models/model_2.py:56-80, called at
 *                                                           quantify_droplets_batch.py:52, and the
 *                                                           `> thresh` of quantify_droplets_batch.py:56
 *   dc_conv_tc / dc_stem         the nn.Conv2d / ConvTranspose2d / BatchNorm2d / ReLU /
 *                                max_pool2d / cat / sigmoid calls inside that forward
 *                                (models/model_2.py:20-32,40-54,58-80), one layer at a time
 *   dc_rolling_ball              rolling_ball_correction_rgb  utils/data_loader.py:11-24
 *   dc_resize_linear_u8          the two cv2.resize calls     quantify_droplets_batch.py:44, :57
 *   dc_label_stats               quantify                     quantify_droplets_batch.py:81-95
 *   dc_overlay_stencil           cv2.findContours + cv2.drawContours of the overlays
 *                                                           quantify_droplets_batch.py:74-79
 *   dc_roi_mask / dc_radial_density / dc_spatial_density
 *                                generate_roi_mask, get_targets, density_maps of the alternate
 *                                front end                   quantify_pipline.py:44-51, :61-91, :93-97
 *
 * Conventions: every function returns 0 (DC_OK) or a negative DC_E* code and never throws;
 * dc_last_error() gives the message of the calling thread's last failure.  All data pointers
 * are DEVICE pointers owned by the caller (the Python side passes torch tensors' data_ptr()),
 * `stream` is a cudaStream_t passed as void*; no entry point synchronises the device or
 * allocates device memory (workspaces are caller-provided, sized by the *_workspace_bytes
 * queries).  There is no CPU fallback: on a device that is not compute capability 10.x the
 * calls fail with DC_EDEVICE.
 */
#ifndef UNETDC_B200_H
#define UNETDC_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DC_OK 0
#define DC_EINVAL (-1)    /* bad argument / unsupported shape */
#define DC_ECUDA (-2)     /* CUDA runtime or driver error */
#define DC_EDEVICE (-3)   /* not an sm_100 device */
#define DC_ECAPACITY (-4) /* droplet table capacity exceeded (counts are still exact) */
#define DC_EWORKSPACE (-5)

/* Bumped whenever a struct or signature in this header changes, or an entry point's return code for some arguments
 * does; dc_version() returns the value the library was built with and the Python binding refuses to load a library
 * that disagrees. */
#define DC_ABI_VERSION 207

const char* dc_last_error(void);
int dc_version(void);
/* 0 when `device` is usable (compute capability 10.x); fills *sm_count when non-NULL. */
int dc_device_check(int device, int* sm_count);

/* ------------------------------------------------------------------ tensor-core conv layer
 * One 3x3 dilated convolution (padding = dilation) or one 2x2 / stride-2 transposed
 * convolution as an implicit GEMM on tcgen05: A = NHWC bf16 activations fetched by TMA
 * (out-of-bounds zero fill = the padding), B = packed bf16 weights, fp32 accumulators in
 * TMEM, epilogue fused per `epilogue`.
 *
 * Weights (prepared by the host wrapper, BatchNorm already folded in fp32):
 *   DC_KIND_CONV3X3 : w[co][(ky*3 + kx)*Cin + ci]            bf16, row length 9*Cin
 *   DC_KIND_UPCONV2 : w[(a*2 + b)*Cout + co][ci]             bf16, row length Cin
 *                     (a, b = output row / column parity, models/model_2.py:20)
 * bias: fp32 [Cout].
 */
enum { DC_KIND_CONV3X3 = 0, DC_KIND_UPCONV2 = 1 };
enum {
    DC_EPI_STORE = 0,      /* bias (+ReLU) -> bf16 NHWC                                   */
    DC_EPI_STORE_POOL = 1, /* ... and the 2x2/stride-2 max of it -> pool_out               */
    DC_EPI_HEAD = 2,       /* bias+ReLU, then 1x1 conv (Cout -> 1) + sigmoid [+ threshold] */
    DC_EPI_UPSCATTER = 3   /* transposed conv: bias, parity scatter into [B,2H,2W,*]        */
};

typedef struct dc_conv_args {
    int kind;     /* DC_KIND_*  */
    int epilogue; /* DC_EPI_*   */
    int relu;     /* apply max(x, 0) after bias (ignored for UPSCATTER)                    */
    int B, H, W;  /* input (= output for conv3x3) spatial shape of this layer              */
    int Cin, Cout;
    int dilation;
    const void* in;    /* bf16 [B,H,W,in_stride] ; channels [0,Cin) are read               */
    int in_stride;     /* elements between consecutive pixels (>= Cin, multiple of 8)      */
    const void* weight;
    const float* bias;
    void* out;         /* bf16; pixel stride out_stride, channel offset out_offset          */
    int out_stride;
    int out_offset;
    void* pool_out;    /* DC_EPI_STORE_POOL: bf16 [B,H/2,W/2,pool_stride]                  */
    int pool_stride;
    const float* head_w; /* DC_EPI_HEAD: fp32 [Cout]                                        */
    float head_b;
    float thresh;
    float* prob_out;     /* DC_EPI_HEAD: fp32 [B,H,W] or NULL                               */
    uint8_t* mask_out;   /* DC_EPI_HEAD: u8   [B,H,W] {0,1} or NULL                         */
    /* Optional, DC_KIND_CONV3X3 with Cin == Cout == 64, dilation 1, even H and W: the same weights as bf16
     * [2][1152][64] in the order of the skip part (chunk 2) of dc_debug_upfuse_schedule.  When given, the layer
     * runs per output parity class with windows shared between classes (see dc_conv_upfused); NULL = the generic
     * kernels from `weight`. */
    const void* weight_par;
} dc_conv_args_t;

int dc_conv_tc(const dc_conv_args_t* args, void* stream);

/* ConvTranspose2d(128, 64, 2, stride 2) -> cat([up, skip]) -> Conv2d(128, 64, 3, padding 1) + BatchNorm + ReLU
 * (upconv1 + dec1.0, models/model_2.py:29, :76-77) as one layer that never writes `up`: per output parity class
 * (y & 1, x & 1) the two convolutions compose into a 2x2-tap convolution over the transposed conv's INPUT x, with
 * weights the host composes in fp32 and rounds to bf16 once, plus the 3x3 over the skip half.
 *   x     bf16 [B,H,W,x_stride], channels [0,128)
 *   skip  bf16 [B,2H,2W,skip_stride], channels [0,64) from the pointer (it may point into a channel slice)
 *   weight bf16 [2][2176][64]: 64-input-channel rows in the order the kernel's MMA schedule consumes them, one half per
 *         CTA of a pair (dc_debug_upfuse_schedule below lists the MMAs; unet_dc_segmentation_b200/model.py pack_upfused
 *         is the packer): the composed 2x2 taps over x per output parity class cls = (y & 1)*2 + (x & 1), then the
 *         skip half of the 3x3 weights
 *   bias9 fp32 [9][64]: row (row class * 3 + col class), class 0 / 1 / 2 = first / interior / last output row
 *         (column): the conv bias plus the transposed conv's bias through the taps that lie inside the image
 *   out   bf16 [B,2H,2W,out_stride] at channel out_offset. */
typedef struct dc_upfuse_args {
    int B, H, W;
    const void* x;
    int x_stride;
    const void* skip;
    int skip_stride;
    const void* weight;
    const float* bias9;
    int relu;
    void* out;
    int out_stride;
    int out_offset;
    /* C: x has 2C channels, skip and the output C.  0 or 64 = the level-1 layer described above.  128 / 256 / 512
     * (upconv{2,3,4} + dec{2,3,4}.0): the tile's parity classes are walked in passes of 256 / min(C, 256) classes, and
     *   weight      bf16 [class group][n-tile][2 CTAs][2C/64 x chunks][4 taps][classes of the group x BN/2 rows][64]
     *   weight_skip bf16 [n-tile][2 CTAs][C/64 chunks][9 taps][BN/2 rows][64]        (BN = min(C, 256); row = output
     *               channel n-tile * BN + CTA * BN/2 + r;  model.py pack_upfused_wide is the packer)
     *   bias9       fp32 [9][C] */
    int channels;
    const void* weight_skip;
} dc_upfuse_args_t;

int dc_conv_upfused(const dc_upfuse_args_t* args, void* stream);
/* Host only (no GPU needed): the MMA schedule of dc_conv_upfused, 5 ints per MMA in issue order = {chunk (0, 1: x
 * channels [64 chunk, 64 chunk + 64); 2: skip), window row, window column, first accumulator slot, slots (1, 2 or 4)};
 * accumulator slot s holds output parity class s ^ (s >> 1).
 * Class cls of an MMA on window (r, c) uses tap (r - py, c - px) of its 2x2 (x chunks) or 3x3 (skip) weights; its B
 * operand is the classes' [64 co][64 ci] tiles stacked, rows [0, N/2) in the first CTA's half of the blob and
 * [N/2, N) in the second's.  Returns the number of MMAs (38) or a negative DC_E* code. */
int dc_debug_upfuse_schedule(int* out, int cap);
/* TEST / MEASUREMENT AID, never called on the product path: which windows dc_conv_upfused shares between classes
 * (0, the default: N = 256 / 128 / 64 MMAs as the windows allow; 1: no sharing, one N = 64 MMA per class and tap;
 * 2: sharing in the x chunks only; 3: only the four-class windows).  Weights must be packed for the mode in force
 * (dc_debug_upfuse_schedule follows it).  Process-wide. */
int dc_debug_set_upfuse_mode(int mode);

/* TEST AID, never called on the product path: pins which kernel family dc_conv_tc picks for layers that have a
 * choice, so that the fallback kernels stay under test.  AUTO (the default): CTA-pair halo kernel where it fits,
 * else single-CTA halo, else per-tap.  Process-wide; not thread-safe against concurrent launches. */
enum { DC_CONV_FAMILY_AUTO = 0, DC_CONV_FAMILY_NO_PAIR = 1, DC_CONV_FAMILY_GENERIC = 2 };
int dc_debug_set_conv_family(int family);

/* First layer (Cin = 3, models/model_2.py:10 first conv) + BatchNorm + ReLU on tcgen05: the im2col tile is
 * built in shared memory by producer warps (K = 27 -> 32, or 9 -> 16 for grayscale where the three identical
 * channels are folded into one), operands in bf16, fp32 accumulation.
 * in_kind 0: fp32 NCHW [B,3,H,W] (the nn.Module contract; rounded to bf16)
 * in_kind 1: u8 planar [B,H,W]   grayscale, replicated to 3 channels, scaled by 1/255 (exact: u8 fits bf16,
 *            the 1/255 is folded into the weights)
 * in_kind 2: u8 HWC    [B,H,W,3] scaled by 1/255               (quantify_droplets_batch.py:41-45)
 * weight fp32 [64][3][3][3] (BN folded), bias fp32 [64]; out bf16 NHWC. */
typedef struct dc_stem_args {
    int in_kind;
    int B, H, W;
    int Cout; /* must be 64 */
    int dilation;
    const void* in;
    const float* weight;
    const float* bias;
    void* out;
    int out_stride;
    int out_offset;
} dc_stem_args_t;

int dc_stem(const dc_stem_args_t* args, void* stream);

/* ------------------------------------------------------------------ whole network */
typedef struct dc_model dc_model_t;

/* Layer order of the 23 weight blobs handed to dc_model_create (names = state_dict prefixes):
 *  0 enc1.0 (stem, fp32)  1 enc1.3  2 enc2.0  3 enc2.3  4 enc3.0  5 enc3.3  6 enc4.0  7 enc4.3
 *  8 bottleneck.0  9 bottleneck.3  10 upconv4  11 dec4.0  12 dec4.3  13 upconv3  14 dec3.0
 * 15 dec3.3  16 upconv2  17 dec2.0  18 dec2.3  19 upconv1  20 dec1.0  21 dec1.3
 * 22 out_conv (fp32 weight [64], bias[1]) */
#define DC_NUM_LAYERS 23
typedef struct dc_model_desc {
    const void* weight[DC_NUM_LAYERS];
    const float* bias[DC_NUM_LAYERS];
    int dilations[5]; /* enc1..enc4, bottleneck: (1,2,4,8,16) for UNetDC, all 1 for plain UNet */
    int base_channels; /* 64 */
    /* UNetDC(in_channels, out_channels), models/model_2.py:6.  (3, 1) -- what quantify_droplets_batch.py:35 builds -- is
     * the fused fast path.  Other counts run the same tensor-core layers around two plain kernels: in_channels != 3
     * (1..64): the fp32 NCHW input is converted to bf16 NHWC zero-padded to 64 channels and enc1.0 runs as an ordinary
     * 3x3 layer, so weight[0] is then bf16 [64][9*64] in the DC_KIND_CONV3X3 layout (input channels padded with zeros)
     * and only in_kind 0 is accepted; out_channels != 1 (1..64): dec1.3 stores its bf16 feature map and a 1x1 kernel
     * applies out_conv (weight[22] fp32 [out][64], bias[22] fp32 [out]) + sigmoid.  0 means the default. */
    int in_channels;
    int out_channels;
    /* Optional: upconv1 + dec1.0 as one launch (dc_conv_upfused).  fused_weight1 / fused_bias1 in the layouts of
     * dc_upfuse_args.weight / .bias9; NULL = run the two layers separately from weight[19], weight[20]. */
    const void* fused_weight1;
    const float* fused_bias1;
    /* Optional, levels 2..4 ([0] = upconv2 + dec2.0, ...): dc_upfuse_args.weight / .weight_skip / .bias9 for
     * channels = 128, 256, 512; a NULL fused_wide_x[i] runs the two layers separately. */
    const void* fused_wide_x[3];
    const void* fused_wide_s[3];
    const float* fused_wide_b[3];
    /* Optional: weights of enc1.3 ([0]) and dec1.3 ([1]) in the dc_conv_args.weight_par layout (used when
     * dilations[0] == 1); NULL = weight[1] / weight[21] through the generic kernels. */
    const void* par_weight[2];
} dc_model_desc_t;

int dc_model_create(dc_model_t** out, int device, const dc_model_desc_t* desc);
int dc_model_destroy(dc_model_t* m);
int dc_forward_workspace_bytes(const dc_model_t* m, int B, int H, int W, size_t* bytes);
/* in_kind as dc_stem_args (in_kind 0: fp32 [B,in_channels,H,W]).  prob_out fp32 [B,out_channels,H,W] and/or mask_out
 * u8 [B,H,W] may be NULL.  mask = prob[:, 0] > thresh (fp32 compare, quantify_droplets_batch.py:56). H, W multiples
 * of 16.  Shape limits: the batch has no limit of its own (B > 65535 runs, also through the in_channels /
 * out_channels != (3, 1) kernels); each layer needs fewer than 2^31 output tiles (DC_EINVAL otherwise).  Element
 * offsets are 64-bit: a level-0 activation or the unfused [B,H,W,128] skip concatenation may exceed 2^31 elements. */
int dc_forward(dc_model_t* m, int in_kind, const void* in, int B, int H, int W, float thresh, float* prob_out,
               uint8_t* mask_out, void* workspace, size_t workspace_bytes, void* stream);
/* number of kernels one dc_forward launches (for bench accounting) */
int dc_forward_num_launches(const dc_model_t* m);
/* Measurement aid: the same forward with a CUDA event between consecutive launches; synchronises the
 * stream and fills launch_ms[dc_forward_num_launches()] (launch order = the layer order above, with
 * out_conv fused into the last one).  Not used on the product path. */
int dc_forward_profile(dc_model_t* m, int in_kind, const void* in, int B, int H, int W, float thresh, float* prob_out,
                       uint8_t* mask_out, void* workspace, size_t workspace_bytes, void* stream, float* launch_ms);

/* ------------------------------------------------------------------ rolling-ball correction
 * Per plane: opening with the radius x radius ellipse of cv2.getStructuringElement, saturating
 * subtract, min-max stretch to 0..255 (utils/data_loader.py:11-24).
 * in/out: u8, `planes` = B*C planes addressed as in[(b*H*W + y*W + x)*C + c] (HWC interleaved;
 * C = 1 is planar grayscale). */
typedef struct dc_rolling_ball_args {
    const uint8_t* in;
    uint8_t* out;
    int B, H, W, C;
    int radius;
    void* workspace;
    size_t workspace_bytes;
} dc_rolling_ball_args_t;

/* Radius 1..dc_rolling_ball_tiled_max_radius() (170): the tiled chord kernel (haloed tiles in shared memory).
 * Larger radii, up to dc_rolling_ball_max_radius() (2047): the banded pass (rectangle decomposition of the ellipse,
 * full rows of a band of output rows in shared memory), which takes rows of at most
 * DC_ROLLING_BALL_BANDED_MAX_WIDTH pixels and returns DC_EINVAL for wider ones.  Both run three kernels inside the
 * same workspace, allocate nothing, do not synchronise, and allow out == in. */
#define DC_ROLLING_BALL_BANDED_MAX_WIDTH 32768
int dc_rolling_ball_workspace_bytes(int B, int H, int W, int C, size_t* bytes);
/* Shape limits of all three entry points (DC_EINVAL otherwise): B*C <= 65535 planes, H*W < 2^31 pixels per plane.
 * The tiled kernel puts rows of tiles (128, 64 or 32 rows, by radius) in gridDim.y; a frame with more than 65535 rows
 * of tiles (H > 8388480 at radius 50) runs the banded pass, bit for bit the same result. */
int dc_rolling_ball(const dc_rolling_ball_args_t* args, void* stream);
/* The tiled kernel alone: radius 1..dc_rolling_ball_tiled_max_radius(), at most 65535 rows of tiles; returns
 * DC_EINVAL where dc_rolling_ball would hand the frame to the banded pass. */
int dc_rolling_ball_tiled(const dc_rolling_ball_args_t* args, void* stream);
/* The banded pass at any radius 1..dc_rolling_ball_max_radius(), also where dc_rolling_ball would run the tiled
 * kernel (the two agree bit for bit); same arguments and workspace as dc_rolling_ball.  Any height (row bands go in
 * gridDim.x); rows of at most DC_ROLLING_BALL_BANDED_MAX_WIDTH pixels. */
int dc_rolling_ball_banded(const dc_rolling_ball_args_t* args, void* stream);
/* Largest `radius` dc_rolling_ball accepts: 2047, an element half as wide as a 4096^2 frame. */
int dc_rolling_ball_max_radius(void);
/* Largest `radius` dc_rolling_ball runs with the tiled kernel (the haloed tile of the element has to fit in shared
 * memory); above it, the banded pass. */
int dc_rolling_ball_tiled_max_radius(void);
/* TEST AID (host only, no GPU needed): dumps the chord plan the kernel would run for `radius` with tiles of
 * `tile_h` rows; returns the number of ints written (layout: csrc/morph.cu) or a negative DC_E* code. */
int dc_debug_rolling_ball_plan(int radius, int tile_h, int* out, int cap);
/* TEST AID (host only, no GPU needed): dumps the rectangles of the banded pass for `radius`:
 * [k, K, piece], then {ya, yb, xa, xb} (rows and columns relative to the output pixel) for each of the K rectangles
 * in walk order, widest chord first; `piece` is the run of pixels one thread scans.  Returns the number of ints
 * written or a negative DC_E* code. */
int dc_debug_rolling_ball_bands(int radius, int* out, int cap);

/* ------------------------------------------------------------------ bilinear resize (u8)
 * The two cv2.resize calls of quantify_droplets_batch.py:44 (frame -> IMG_SIZE x IMG_SIZE) and :57 (mask -> original
 * size).  Both pass their interpolation flag in cv2.resize's `dst` slot, so both are OpenCV's default INTER_LINEAR
 * on 8-bit data (11-bit fixed point); this entry point reproduces that bit for bit.
 * in: u8 [B, src_h, src_w, C] interleaved (C = 1 or 3); out: u8 [B, dst_h, dst_w, C]. */
typedef struct dc_resize_args {
    const uint8_t* in;
    uint8_t* out;
    int B, C;
    int src_h, src_w;
    int dst_h, dst_w;
} dc_resize_args_t;

/* Shape limits (DC_EINVAL otherwise): B <= 65535 and dst_h <= 65535 (grid dimensions). */
int dc_resize_linear_u8(const dc_resize_args_t* args, void* stream);

/* ------------------------------------------------------------------ labelling + droplet table
 * quantify() of quantify_droplets_batch.py:81-95 for a batch of masks: 4-connected labelling,
 * min_area filter, consecutive relabelling in raster order of first pixel, per-droplet
 * area / centroid / equivalent diameter (+ micron columns when px_per_um > 0).
 * Table row r of image b lives at index b*capacity + r (label = r + 1). */
typedef struct dc_label_args {
    const uint8_t* mask; /* u8 [B,H,W], non-zero = foreground */
    int B, H, W;
    int64_t min_area;
    double px_per_um;    /* <= 0: micron columns not written */
    int32_t* labels_out; /* int32 [B,H,W] or NULL */
    int capacity;        /* table rows per image */
    int32_t* counts;     /* int32 [B]: droplets kept per image (exact even on overflow) */
    int64_t* area;       /* [B*capacity] */
    double* centroid0;   /* row  */
    double* centroid1;   /* col  */
    double* eq_diam;
    double* area_um2;    /* may be NULL when px_per_um <= 0 */
    double* diam_um;
    void* workspace;
    size_t workspace_bytes;
} dc_label_args_t;

int dc_label_workspace_bytes(int B, int H, int W, size_t* bytes);
/* Shape limits (DC_EINVAL otherwise): B <= 65535, H*W < 2^31, H <= 65535 * 128 (rows of 128-row tiles in gridDim.y). */
int dc_label_stats(const dc_label_args_t* args, void* stream);

/* ---- overlay stencil --------------------------------------------------------------------------
 * stencil[b,y,x] = 1 exactly where
 *     cnts, _ = cv2.findContours(mask, cv2.RETR_EXTERNAL, cv2.CHAIN_APPROX_SIMPLE)
 *     cv2.drawContours(img, cnts, -1, (0, 255, 0), 2)        (quantify_droplets_batch.py:76-77)
 * changes img, else 0: the caller paints those pixels (0, 255, 0) in the BGR frame it read (qdb:75,78).
 * Only top-level borders (droplets nested inside a hole of another are not outlined), thickness 2 as
 * OpenCV rasterises it.  mask: u8 [B,H,W], non-zero = foreground.  Bit-exact against OpenCV 4.x. */
typedef struct dc_overlay_args {
    const uint8_t* mask;
    int B, H, W;
    uint8_t* stencil;    /* u8 [B,H,W], {0,1} */
    void* workspace;
    size_t workspace_bytes;
} dc_overlay_args_t;

int dc_overlay_workspace_bytes(int B, int H, int W, size_t* bytes);
/* Shape limits as dc_label_stats: B <= 65535, H*W < 2^31, H <= 65535 * 128. */
int dc_overlay_stencil(const dc_overlay_args_t* args, void* stream);

/* ---- density maps of quantify_pipline.py (the reference's alternate front end) ---------------------------
 * All three are bit-exact against the OpenCV / numpy / scipy calls they replace.
 *
 * dc_roi_mask: generate_roi_mask(img) (quantify_pipline.py:44-51: RGB2GRAY, GaussianBlur 15x15, Otsu,
 *   15x15 close, 15x15 open, > 0) and the centroid of quantify_pipline.py:133-136
 *   (cx = int(m10/m00), cy = int(m01/m00) of cv2.moments, image centre when the mask is empty).
 *   rgb: u8 [B,H,W,3]; roi: u8 [B,H,W] {0,1}; centroid: int32 [B][2] = (cy, cx). */
typedef struct dc_roi_args {
    const uint8_t* rgb;
    int B, H, W;
    uint8_t* roi;
    int* centroid;
    void* workspace;
    size_t workspace_bytes;
} dc_roi_args_t;

int dc_roi_workspace_bytes(int B, int H, int W, size_t* bytes);
/* Shape limits (DC_EINVAL otherwise): B <= 65535, H <= 65535, H*W < 2^31. */
int dc_roi_mask(const dc_roi_args_t* args, void* stream);

/* dc_radial_density: get_targets(mask, roi, nb_layers, cy, cx) (quantify_pipline.py:61-91).  The droplet
 *   centroids are the centroid0 / centroid1 / counts columns dc_label_stats wrote for the same masks with
 *   min_area = 1 (the reference labels the mask again without a size filter, :66-68).  out: f32 [B,H,W]. */
typedef struct dc_radial_args {
    const uint8_t* roi;
    int B, H, W;
    const int* centroid;        /* [B][2] = (cy, cx) */
    const int* counts;          /* [B] */
    const double* centroid0;    /* [B,capacity] row */
    const double* centroid1;    /* [B,capacity] col */
    int capacity;
    int nb_layers;              /* 1..64; the reference uses 10 (:138) */
    float* out;
    void* workspace;
    size_t workspace_bytes;
} dc_radial_args_t;

int dc_radial_workspace_bytes(int B, size_t* bytes);
/* Shape limits (DC_EINVAL otherwise): B <= 65535, H*W < 2^31. */
int dc_radial_density(const dc_radial_args_t* args, void* stream);

/* dc_spatial_density: density_maps(mask, roi, kernel_size) (quantify_pipline.py:93-97):
 *   100 * gaussian_filter(mask) / (gaussian_filter(roi) + 1e-5), scipy.ndimage.gaussian_filter on float32 with
 *   mode='reflect'.  weights: HOST pointer to the 2*radius+1 normalised f64 taps scipy builds for the sigma
 *   (sigma = kernel_size / 6, radius = int(4*sigma + 0.5)); read during the call.  out: f32 [B,H,W]. */
#define DC_GAUSS_MAX_RADIUS 64
typedef struct dc_spatial_args {
    const uint8_t* mask;
    const uint8_t* roi;
    int B, H, W;
    int radius;
    const double* weights;
    float* out;
    void* workspace;
    size_t workspace_bytes;
} dc_spatial_args_t;

int dc_spatial_workspace_bytes(int B, int H, int W, size_t* bytes);
/* Shape limits (DC_EINVAL otherwise): B <= 65535, H <= 65535 * 16 (rows of 16-row tiles in gridDim.y). */
int dc_spatial_density(const dc_spatial_args_t* args, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* UNETDC_B200_H */
