/*
 * irmv_cabi.h -- C ABI of the B200-native per-frame armor pipeline (libirmv_b200.so).
 *
 * This is the drop-in boundary: plain pointers and sizes, no C++/torch types.  The C++ classes in
 * include/irmv_detection/{yolo_engine,pnp_solver}.hpp keep the reference's signatures and call
 * these functions; the Python mirror (irmv_detection_b200/) binds the same symbols with ctypes.
 * Every function returns 0 on success and a non-zero code on failure (irmv_last_error() then
 * holds a message); nothing throws across this boundary and nothing falls back to the CPU.
 *
 * Reference interfaces replaced (paths into the reference tree, illini-robomaster/irmv_detection):
 *   irmv_engine_create        <- YoloEngine::YoloEngine          src/yolo_engine.cpp:24-117
 *   irmv_engine_destroy       <- YoloEngine::~YoloEngine         src/yolo_engine.cpp:119-135
 *   irmv_engine_src_buffer    <- get_src_image_buffer()          include/irmv_detection/yolo_engine.hpp:35
 *   irmv_engine_rotated_image <- get_rotated_image()             include/irmv_detection/yolo_engine.hpp:34
 *   irmv_engine_detect        <- YoloEngine::detect()            src/yolo_engine.cpp:153-177
 *                                (graph launch :164, sync :165, parse_output :202-220)
 *   irmv_engine_profile_ms    <- get_profiling_time()            include/irmv_detection/yolo_engine.hpp:33
 *   irmv_preprocess           <- YoloEngine::preprocess()        src/yolo_engine.cpp:179-200 (NPP K1-K4)
 *   irmv_nms                  <- EfficientNMS_TRT inside the engine  src/yolo_engine.cpp:33,53-57
 *   irmv_pnp_create           <- PnPSolver::PnPSolver            src/pnp_solver.cpp:7-34
 *   irmv_pnp_solve            <- PnPSolver::solvePnP             src/pnp_solver.cpp:36-52
 *   irmv_pnp_distance_to_center <- calculateDistanceToCenter     src/pnp_solver.cpp:54-59
 *   irmv_engine_fetch_keypoints: keypoint variant of the detector (reference README.md:12,16)
 *   irmv_extract_armors       <- IrmDetector::extract_armors     src/irm_detector.cpp:292-355
 *                                (+ Light / Armor constructors, include/irmv_detection/armor.hpp:11-77)
 *   irmv_engine_detect_batch / irmv_pnp_solve_batch: batch forms of the same calls for the
 *   multi-frame configs of BASELINE.json (the reference is batch-1 only).
 */
#ifndef IRMV_CABI_H_
#define IRMV_CABI_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define IRMV_NET_SIZE 640      /* src/yolo_engine.cpp:98-99,189-198 */
#define IRMV_NUM_CLASSES 14    /* include/irmv_detection/armor.hpp:7 */
#define IRMV_CLASS_UNKNOWN 14

/* channel order of the source buffer */
enum {
  IRMV_CH_PASSTHROUGH = 0, /* reference: bytes go to the net in buffer order */
  IRMV_CH_SWAP_RB = 1,
  IRMV_CH_BAYER_RGGB = 2,
  IRMV_CH_BAYER_BGGR = 3,
  IRMV_CH_BAYER_GRBG = 4,
  IRMV_CH_BAYER_GBRG = 5
};

/* MindVision frame header field tSdkFrameHead.uiMediaType (reference mvsdk/include/CameraDefine.h:609-627;
 * 8-bit Bayer codes :733-736, packed RGB8 / BGR8 :771-772) -> IRMV_CH_* for a raw sensor frame handed to the
 * engine instead of the vendor ISP's RGB8 output (reference src/mv_camera.cpp:64,96).  The vendor names a
 * pattern by the first two pixels of the first row: BAYRG = R G / G B = RGGB, BAYGR = GRBG, BAYGB = GBRG,
 * BAYBG = BGGR.  Covers the 8-bit formats: returns -1 for everything else, including the 10/12-bit Bayer formats
 * the engine ingests through raw_format (irmv_source_format_from_media_type maps those). */
#define IRMV_MV_MEDIA_TYPE_BAYGR8 0x01080008u
#define IRMV_MV_MEDIA_TYPE_BAYRG8 0x01080009u
#define IRMV_MV_MEDIA_TYPE_BAYGB8 0x0108000Au
#define IRMV_MV_MEDIA_TYPE_BAYBG8 0x0108000Bu
#define IRMV_MV_MEDIA_TYPE_RGB8 0x02180014u
#define IRMV_MV_MEDIA_TYPE_BGR8 0x02180015u
int irmv_chan_order_from_media_type(uint32_t mv_media_type);

/* Format of the raw samples of a Bayer source (irmv_engine_config.raw_format).  Frames are row-major without line
 * padding.  RAW_8: one byte per sample (W*H bytes, the default).  RAW_10 / RAW_12: one little-endian uint16 per
 * sample, the value in the low 10 / 12 bits; the bits above are ignored (W*H*2 bytes).  RAW_12_PACKED: two
 * horizontally adjacent samples in three bytes, B0 = p0[11:4], B1 = p1[3:0] << 4 | p0[3:0], B2 = p1[11:4]
 * (W*H*3/2 bytes, W even) -- the GigE Vision "BayerXX12Packed" layout the vendor's media-type numbering follows,
 * taken from that definition and not checked against bytes from a real camera. */
enum { IRMV_RAW_8 = 0, IRMV_RAW_10 = 1, IRMV_RAW_12 = 2, IRMV_RAW_12_PACKED = 3 };
/* The vendor header's MONO | occupancy | id codes of the 10-bit, 12-bit and 12-bit packed Bayer formats. */
#define IRMV_MV_MEDIA_TYPE_BAYGR10 0x0110000Cu
#define IRMV_MV_MEDIA_TYPE_BAYRG10 0x0110000Du
#define IRMV_MV_MEDIA_TYPE_BAYGB10 0x0110000Eu
#define IRMV_MV_MEDIA_TYPE_BAYBG10 0x0110000Fu
#define IRMV_MV_MEDIA_TYPE_BAYGR12 0x01100010u
#define IRMV_MV_MEDIA_TYPE_BAYRG12 0x01100011u
#define IRMV_MV_MEDIA_TYPE_BAYGB12 0x01100012u
#define IRMV_MV_MEDIA_TYPE_BAYBG12 0x01100013u
#define IRMV_MV_MEDIA_TYPE_BAYGR12_PACKED 0x010C002Au
#define IRMV_MV_MEDIA_TYPE_BAYRG12_PACKED 0x010C002Bu
#define IRMV_MV_MEDIA_TYPE_BAYGB12_PACKED 0x010C002Cu
#define IRMV_MV_MEDIA_TYPE_BAYBG12_PACKED 0x010C002Du
/* Media type -> (IRMV_CH_*, IRMV_RAW_*) for every format the engine ingests: the 8-bit Bayer formats, RGB8 and BGR8
 * (raw_format IRMV_RAW_8) and the 10-bit, 12-bit and 12-bit packed Bayer formats.  Returns 0 and fills both outputs,
 * non-zero for anything else (10-bit packed, 16-bit, mono, YUV, planar). */
int irmv_source_format_from_media_type(uint32_t mv_media_type, int32_t *chan_order, int32_t *raw_format);

/* STRETCH = the reference: independent x/y scale, NPP's measured corner-aligned bilinear map
 * (src = dst * src_size/640, no half-pixel offset; pinned in tests/golden/npp_rm_golden.npz).
 * STRETCH_HALF_PIXEL = same stretch with OpenCV-style pixel centres.  LETTERBOX = ultralytics
 * LetterBox (aspect-preserving resize, centred, pad 114), not what the reference does. */
enum { IRMV_RESIZE_STRETCH = 0, IRMV_RESIZE_LETTERBOX = 1, IRMV_RESIZE_STRETCH_HALF_PIXEL = 2 };
enum { IRMV_CONV_TCGEN05 = 0, IRMV_CONV_DIRECT = 1 /* CUDA-core bring-up kernel */ };

/* Same layout as YoloEngine::bbox (include/irmv_detection/yolo_engine.hpp:19-26): 24 bytes. */
typedef struct irmv_bbox {
  float xyxy[4];    /* source-frame pixels (already multiplied by W/640, H/640) */
  float score;
  int32_t class_id; /* 0..13, 14 = UNKNOWN */
} irmv_bbox;

typedef struct irmv_engine_config {
  int32_t src_width;        /* 1280 in the reference node, src/irm_detector.cpp:142-143 */
  int32_t src_height;       /* 1024 */
  int32_t chan_order;       /* IRMV_CH_* */
  int32_t rotate180;        /* 1 = reference (nppiMirror both axes, src/yolo_engine.cpp:182-184) */
  int32_t resize_mode;      /* IRMV_RESIZE_* */
  int32_t quantize_u8;      /* 1 = keep the reference's 8-bit intermediate after the resize */
  int32_t max_batch;        /* frames per detect_batch call; 1 = reference */
  int32_t sub_batch;        /* frames per graph replay (<= max_batch); 0 = pick (min(max_batch, 256)) */
  int32_t num_lanes;        /* concurrent streams replaying sub-batches; 0 = pick */
  int32_t num_slots;        /* pinned source slots for detect(); 3 = the reference's triple buffer */
  int32_t device;           /* CUDA device ordinal */
  int32_t conv_impl;        /* IRMV_CONV_* */
  int32_t max_det;          /* EfficientNMS max_output_boxes, 100 */
  float score_thr;          /* 0.25 */
  float iou_thr;            /* 0.45 */
  int32_t use_graph;        /* 1 = replay captured CUDA graphs (reference behaviour) */
  int32_t reserved[7];      /* reserved[0] != 0: run preprocess and conv0 as separate kernels (the network
                             * input tensor is then materialised and readable as tap "input");
                             * reserved[1] != 0: do not fuse 1x1 convs into their producers (every module
                             * output is then materialised and readable through irmv_engine_read_tensor);
                             * reserved[2] != 0: ShuffleNetV2 variant: one launch per convolution instead of one fused
                             * kernel per unit;
                             * reserved[3] != 0: the neck's 1x1 convs over concat(upsample(a), b) as ONE gather-kernel
                             * launch each instead of two raster-kernel launches (W_a at a's resolution + W_b) */
  int32_t raw_format;       /* IRMV_RAW_*; anything but IRMV_RAW_8 (0, the default) needs a Bayer chan_order, and
                             * IRMV_RAW_12_PACKED an even src_width.  A 10/12-bit engine decodes every frame into an
                             * 8-bit mosaic through its raw table (irmv_engine_set_raw_lut) before anything else reads
                             * it: one extra kernel per replay, counted in the preprocess stage. */
} irmv_engine_config;

/* One armor as IrmDetector::extract_armors builds it (src/irm_detector.cpp:292-355): slot i of a frame
 * belongs to detection i; valid == 0 when the detection's ROI does not hold two light bars that pass
 * the filters.  pts = the PnP image points in PnPSolver::solvePnP's order (src/pnp_solver.cpp:41-44):
 * left.bottom, left.top, right.top, right.bottom, pixels of the rotated source frame. */
typedef struct irmv_armor {
  float pts[8];
  float center[2];   /* Armor::center, include/irmv_detection/armor.hpp:67 */
  float score;       /* Armor::confidence */
  int32_t class_id;  /* Armor::armor_class */
  int32_t size;      /* ArmorSize: 0 SMALL, 1 LARGE */
  int32_t valid;
} irmv_armor;

/* Node parameters of the light / armor filters (src/irm_detector.cpp:152,162-173). */
typedef struct irmv_armor_params {
  int32_t binary_threshold;            /* 150 */
  float light_min_ratio;               /* 0.1  (Light::is_light takes floats, armor.hpp:31) */
  float light_max_ratio;               /* 0.4 */
  float light_max_angle;               /* 40 degrees */
  double min_small_center_distance;    /* 0.8 */
  double max_small_center_distance;    /* 3.2 */
  double min_large_center_distance;    /* 3.2 */
  double max_large_center_distance;    /* 5.5 */
} irmv_armor_params;

/* Per-armor output of IrmDetector::message_callback (src/irm_detector.cpp:213-230): the
 * auto_aim_interfaces/Armor fields the node fills -- pose.position = tvec, pose.orientation = the tf2
 * quaternion (x, y, z, w) of Rodrigues(rvec) (:218-226), distance_to_image_center (:229, the intended
 * computation of src/pnp_solver.cpp:54-59) -- produced by the fused replay. */
typedef struct irmv_pose {
  double position[3];
  double orientation[4];
  double rvec[3];                   /* the solver's rotation vector, for callers that want it */
  float distance_to_image_center;
  int32_t ok;                       /* 1: slot holds a solved armor (detection present, armor found, PnP ok) */
} irmv_pose;

typedef struct irmv_engine irmv_engine;
typedef struct irmv_pnp irmv_pnp;

const char *irmv_last_error(void);
int irmv_version(void);

/* ---- engine -------------------------------------------------------------------------------- */
int irmv_engine_config_default(irmv_engine_config *cfg);
int irmv_engine_create(const char *weights_path, const irmv_engine_config *cfg, irmv_engine **out);
void irmv_engine_destroy(irmv_engine *e);

/* Borrowed, address-stable pinned-host frame slot the camera writes (one frame: src_w*src_h*3 bytes for packed RGB,
 * otherwise the raw_format's frame size). */
uint8_t *irmv_engine_src_buffer(irmv_engine *e, int slot);
/* get_rotated_image() (include/irmv_detection/yolo_engine.hpp:34; the node calls it every frame,
 * src/irm_detector.cpp:183): *view = address-stable pinned buffer holding the rotated packed-RGB frame
 * of `slot` as of the last detect() on it.  The first call turns the feature on (allocates once and
 * rotates the frame still on the device); afterwards every detect() refreshes the buffer itself and
 * this call only returns the pointer -- no allocation, no re-upload, no extra preprocess. */
int irmv_engine_rotated_view(irmv_engine *e, int slot, const uint8_t **view);
/* Same frame copied into dst (packed u8x3). */
int irmv_engine_rotated_image(irmv_engine *e, int slot, uint8_t *dst);
/* Debug: number of device / pinned allocations this library has made in the process so far (tests
 * assert that per-frame calls make none). */
long long irmv_debug_alloc_count(void);
/* Debug: every activation tensor is a zero-padded raster (guard pixels, a zero row per image, a zero column) and every
 * kernel relies on that padding staying zero.  Counts the padding pixels of all activation tensors of the engine that
 * are not zero: 0 after any sequence of calls, anything else is a stray store (the memory check this pool allows). */
int irmv_debug_check_padding(irmv_engine *e, long long *bad_pixels);
/* Debug: CTAs per SM of the camera-case stem kernel as the engine launches it now (with its raw table when one is
 * set), or 0 when its frames go to the generic stem kernel instead. */
int irmv_debug_stem_ctas(irmv_engine *e, int *ctas);

/* One frame from pinned slot `slot`: H2D + graph(preprocess, net, decode, NMS) + D2H + parse. */
int irmv_engine_detect(irmv_engine *e, int slot, irmv_bbox *out, int cap, int *n);
/* nframes <= max_batch contiguous frames; frames_on_device != 0 means a device pointer.
 * out holds nframes*max_det boxes, counts nframes entries. */
int irmv_engine_detect_batch(irmv_engine *e, const uint8_t *frames, int frames_on_device,
                             int nframes, irmv_bbox *out, int *counts);
/* Same, but leaves results on the device and does not synchronise (bench: inputs resident). */
int irmv_engine_enqueue_batch(irmv_engine *e, const uint8_t *frames_dev, int nframes);
int irmv_engine_sync(irmv_engine *e);
int irmv_engine_fetch(irmv_engine *e, int nframes, irmv_bbox *out, int *counts);
double irmv_engine_profile_ms(irmv_engine *e);
/* Cumulative bytes of the host->device and device->host copies the engine has queued. */
int irmv_engine_copy_bytes(irmv_engine *e, unsigned long long *h2d, unsigned long long *d2h);
/* Device time of the last enqueue/detect (CUDA events on the engine's streams), ms. */
double irmv_engine_last_device_ms(irmv_engine *e);
int irmv_engine_kernel_launches(irmv_engine *e, int nframes);
void *irmv_engine_stream(irmv_engine *e);

/* Fuse the pose stage into the replay: after NMS, the four corners of every kept box (scaled by
 * corner_sx/sy from source pixels to the calibration frame) go through the IPPE kernel on the
 * device; poses come back with the detections.  Replaces the per-armor host loop of
 * IrmDetector::message_callback (src/irm_detector.cpp:204-208). */
int irmv_engine_enable_pnp(irmv_engine *e, const double K[9], const double D[5], float corner_sx,
                           float corner_sy);
/* rvecs/tvecs: nframes*max_det*3 doubles; slot i of frame f is valid when i < counts[f]. */
int irmv_engine_fetch_poses(irmv_engine *e, int nframes, double *rvecs, double *tvecs, uint8_t *ok);
/* The whole per-armor message payload (see irmv_pose) of the last synchronous call (ticket < 0) or of a
 * collected pipelined batch: out holds nframes*max_det entries, slot-aligned with the detections. */
int irmv_engine_fetch_armor_poses(irmv_engine *e, int ticket, int nframes, irmv_pose *out);
/* ---- keypoint variant (BASELINE.json configs[2], north_star "armor-keypoint decode") -------------
 * A weight file with 72 convolutions carries the ultralytics Pose branch (kpt_shape [4, 2]: the four
 * armor corners LB, LT, RT, RB per anchor).  The engine then decodes the keypoints of every kept
 * detection ((raw * 2 + grid) * stride) and, with irmv_engine_enable_pnp, solves the pose on them
 * instead of the box corners. */
int irmv_engine_has_keypoints(irmv_engine *e);
/* kpts: nframes*max_det*8 floats {x, y} x 4, source pixels; slot i of frame f is valid when i < counts[f].
 * ticket < 0: the last synchronous call; otherwise a collected pipelined batch. */
int irmv_engine_fetch_keypoints(irmv_engine *e, int ticket, int nframes, float *kpts);

/* ---- light bars -> armors (IrmDetector::extract_armors, src/irm_detector.cpp:292-355) ---------- */
int irmv_armor_params_default(irmv_armor_params *p);
/* Stage entry: nframes frames as the camera wrote them (the kernel reads the rotated view itself),
 * boxes[nframes*max_det] in source pixels with counts[nframes] valid entries per frame (what detect()
 * returns); out[nframes*max_det], slot-aligned with boxes.  prm == NULL: defaults.  Sources up to
 * 32766 x 32766 with 8 * (src_w + 2) * (src_h + 2) < 2^31; larger ones are refused (returns 2). */
int irmv_extract_armors(const uint8_t *frames, int frames_on_device, int nframes, int src_w, int src_h, int chan_order,
                        int rotate180, const irmv_bbox *boxes, const int *counts, int max_det,
                        const irmv_armor_params *prm, int device, irmv_armor *out);
/* Device time (CUDA events around the kernel) of this thread's last irmv_extract_armors call, ms. */
double irmv_extract_armors_last_device_ms(void);
/* Debug (IRMV_ARMOR_PROF set): SM cycles per phase of that call, summed over ROIs:
 * {bitmap, flood, walks + lights, armor, ROIs processed, flood rounds, recording walks, hull + rectangle + light}. */
int irmv_extract_armors_last_profile(unsigned long long out[8]);
/* Fuse the stage into the replay, between NMS and PnP: with irmv_engine_enable_pnp the pose stage then
 * solves on the armor corners (scaled by corner_sx/sy) instead of the box corners, and ok[] is 0 for
 * detections without an armor -- the whole of message_callback's per-frame work
 * (src/irm_detector.cpp:181-208) in one graph.  Refuses (returns 2) an engine whose source size the
 * stage does not take (see irmv_extract_armors). */
int irmv_engine_enable_armors(irmv_engine *e, const irmv_armor_params *prm);
/* out: nframes*max_det armors of the last detect/detect_batch/sync (ticket < 0) or of a collected
 * pipelined batch (its ticket). */
int irmv_engine_fetch_armors(irmv_engine *e, int ticket, int nframes, irmv_armor *out);

/* Raw-domain colour stage for Bayer sources: lut = [3][2^b] bytes (R, G, B sites) for a b-bit raw_format -- [3][256]
 * for IRMV_RAW_8, [3][1024] for IRMV_RAW_10, [3][4096] for IRMV_RAW_12 and IRMV_RAW_12_PACKED -- or NULL.
 * Applied by every kernel that reads the raw frame: stem / preprocess, rotated view, fused armor stage.
 * A raw sample s at sensor position (y, x) -- frame coordinates as the camera wrote them, before rot180 -- is read
 * as lut[c][s], c = the colour of that site under the engine's pattern (both green sites use lut[1]): the engine
 * with table L on frames F returns what it returns without a table on the frames L(F).  One table covers black
 * level, white-balance gains and a tone curve; the caller's frames are never written.  Non-zero (irmv_last_error)
 * for a packed RGB/BGR source or while pipelined batches are in flight.
 * 8-bit engines: NULL = off, the default.  The first non-NULL call allocates the device table, later calls rewrite
 * it; switching between off and on drops the captured graphs.
 * 10/12-bit engines: the table maps a b-bit sample to the 8-bit value the rest of the pipeline sees; NULL (and the
 * default) is the shift s >> (b - 8).  Every call rewrites the table allocated at create: no allocation, the
 * captured graphs stay. */
int irmv_engine_set_raw_lut(irmv_engine *e, const uint8_t *lut);

/* Colour-correction stage for Bayer sources: m = 3x3 int16 matrix (row-major, units of 1/1024: identity is 1024 * I)
 * and tone_lut = [3][256] output tone table (R, G, B) or NULL (identity); m == NULL switches the stage off (the
 * default), and then tone_lut must be NULL too.  Applied by every kernel that demosaics the raw frame (stem /
 * preprocess, rotated view, fused armor stage) to every demosaiced pixel -- after the raw table (or the 10/12-bit
 * decode), before rot180 and resize -- so it is the u8 RGB frame the network input, the rotated view and the armor
 * stage's gray values are computed from:
 *   v_c = sum_k m[c][k] * in_k,  out_c = tone_lut[c][clamp((v_c + 512) >> 10, 0, 255)]   (integer, arithmetic shift)
 * The Bayer engine with matrix M and tone T on frames F returns what an otherwise identical IRMV_CH_PASSTHROUGH
 * engine without it returns on the packed frames T(M(demosaic(F))).  A saturation gain is one such matrix; with the
 * ISP order -- black level and gains in the raw table at gamma 1, then the matrix, then gamma in tone_lut -- the
 * engine reproduces the camera ISP's colour chain (auto white balance: irmv_engine_set_auto_white_balance).  Non-zero (irmv_last_error) for a
 * packed RGB/BGR source (its ISP has already applied a matrix), for a tone table without a matrix, or while pipelined
 * batches are in flight.  Works for every raw_format.  The first non-NULL call allocates the device block, later
 * calls rewrite it in place (no allocation, the captured graphs stay); switching between off and on drops the
 * captured graphs. */
int irmv_engine_set_color_matrix(irmv_engine *e, const int16_t m[9], const uint8_t *tone_lut);

/* Automatic white balance for Bayer sources, per frame and stateless: the gains applied to a frame are a function of
 * that frame alone (raw_lut.awb_statistics / awb_gains / awb_matrix are the definition).  The input is the 8-bit
 * mosaic the demosaic reads (IRMV_RAW_8: after the raw table; 10/12-bit: the decoded mosaic), in sensor coordinates.
 * Quad (i, j) covers rows 2i, 2i+1 and columns 2j, 2j+1 (i < H/2, j < W/2); it is clipped if a sample is > clip_level,
 * else dark if a sample is < dark_level, else counted.  Over the counted quads SR = sum R, SG = sum (Gr + Gb),
 * SB = sum B; with A = (2 SR, SG, 2 SB) the Q10 gains are g_c = min((1024 max(A) + A_c / 2) / A_c, gain_max_q10), so
 * the brightest channel keeps 1024.  A frame with counted < min_quads or an empty channel keeps (1024, 1024, 1024)
 * and valid = 0.  The gains are applied by the colour-correction stage: frame F is demosaiced with
 *   M_F[r][k] = clamp_int16((M[r][k] * g_k + 512) >> 10)   (M = the set_color_matrix matrix, or 1024 * I)
 * and the tone table T of set_color_matrix (or identity).  So set_color_matrix(M_F, T) with AWB off reproduces what
 * AWB did to F exactly: fetch the gains, compose them and switch AWB off to lock the white balance.  ISP order: the
 * raw table takes black level only, then AWB, then the matrix, then tone. */
typedef struct irmv_awb_params {
  int32_t dark_level;    /* quads with a sample below this are not counted (default 8)    */
  int32_t clip_level;    /* quads with a sample above this are not counted (default 250)  */
  int32_t min_quads;     /* fewer counted quads: gains 1, valid 0 (default 4096)          */
  int32_t gain_max_q10;  /* upper clamp of every gain, >= 1024 (default 4096)             */
} irmv_awb_params;
typedef struct irmv_awb {            /* one per frame, what was applied to that frame */
  uint64_t sum[3];                   /* SR, SG (both green sites), SB over counted quads */
  uint32_t counted, dark, clipped;   /* quads; dark/clipped are what a host exposure loop needs */
  int32_t valid;
  int32_t gain_q10[3];
  int32_t reserved;
} irmv_awb;
int irmv_awb_params_default(irmv_awb_params *p);
/* p == NULL switches the stage off (the default).  Refused: a packed RGB/BGR source (returns 2), parameters outside
 * 0 <= dark_level <= clip_level <= 255, min_quads >= 1, 1024 <= gain_max_q10 <= 32767 (returns 1), pipelined
 * batches in flight (returns 5).  Every replay then runs one statistics kernel first and every kernel that demosaics
 * the raw frame reads its frame's own block.  The first call that switches it on allocates; later calls rewrite the
 * parameters in place (no allocation, the captured graphs stay), and so does a set_color_matrix update; switching
 * between off and on drops the captured graphs.  Per-frame calls allocate nothing. */
int irmv_engine_set_auto_white_balance(irmv_engine *e, const irmv_awb_params *p);
/* out: nframes records of the last detect/detect_batch/sync (ticket < 0) or of a collected pipelined batch (its
 * ticket).  An error with the stage off or for a call that ran without it. */
int irmv_engine_fetch_white_balance(irmv_engine *e, int ticket, int nframes, irmv_awb *out);

/* Pipelined hand-off for host-resident batches -- the B200 form of the overlap the reference gets
 * from its TripleBuffer (camera thread fills the next slot while detect() runs on the previous one,
 * reference README.md:60-63, src/irm_detector.cpp:68-72).  submit queues H2D copy (dedicated copy
 * stream) + pipeline + D2H of the results and returns; collect waits for that batch and parses it
 * like detect_batch (rvecs/tvecs/ok may be null).  At most three batches in flight; collect in order.
 * The hand-off is checked: a fourth submit before a collect, a ticket that is not in flight (stale,
 * duplicate, never issued), an out-of-order collect, and any synchronous entry point (detect,
 * detect_batch, enqueue_batch, rotated image) while batches are in flight return an error.
 * Host batches are replayed in chunks of at most 128 frames whatever sub_batch is (a chunk starts as soon as its
 * own frames have landed, under the copy of the next one); synchronous detect_batch calls with more than 128 host
 * frames take the same route.  Results do not depend on the chunking. */
int irmv_engine_submit_batch(irmv_engine *e, const uint8_t *frames_host, int nframes, int *ticket);
int irmv_engine_collect(irmv_engine *e, int ticket, irmv_bbox *out, int *counts, double *rvecs, double *tvecs,
                        uint8_t *ok);
/* One eager replay of min(nframes, sub_batch) device-resident frames with CUDA events between
 * stages: ms = {preprocess, convolutions, decode+NMS, PnP, total}.  Returns frames profiled. */
int irmv_engine_profile_stages(irmv_engine *e, const uint8_t *frames_dev, int nframes, float ms[5]);

/* Debug/tuning: per-tile clock64 stamps of CTA 0 for GEMM `op_index` (see engine.cu). */
/* Debug: text description of the network stage's kernels in issue order (one line per launch). */
int irmv_engine_describe_ops(irmv_engine *e, char *buf, int cap);
/* Debug: tiling plan / kernel instantiation of every network-stage launch for a replay of nframes frames. */
int irmv_engine_describe_plans(irmv_engine *e, int nframes, char *buf, int cap);
/* Debug: per-kernel CUDA-event times (ms) of the network stage of one eager replay. */
int irmv_engine_profile_ops(irmv_engine *e, const uint8_t *frames_dev, int nframes, float *ms, int cap);
int irmv_engine_trace_conv(irmv_engine *e, int op_index, int nframes, long long *out, int cap_tiles,
                           float *kernel_ms);

/* Parity taps: raw activations of the last run.  name: "input" (preprocessed, NHWC8 FP16),
 * "box0".."box2" (NHWC64), "cls0".."cls2" (NHWC16), "boxes" (f32 [A,4]), or a module tap
 * ("m0".."m21").  Copies up to cap_bytes to dst (host); dims receives {B,H,W,C,elem_size}. */
int irmv_engine_read_tensor(irmv_engine *e, const char *name, void *dst, int64_t cap_bytes,
                            int32_t dims[5]);
/* Kept flat indices (anchor*nc+class) of frame i of the last run, for bit-exact NMS parity. */
int irmv_engine_read_kept_indices(irmv_engine *e, int frame, int32_t *idx, int cap, int *n);

/* ---- stage entry points (each is what the engine runs, exposed for parity tests) ------------ */
/* src: host u8 frames [n][H][W][3] (or [n][H][W] Bayer); dst: host FP16 [n][640][640][8] NHWC. */
int irmv_preprocess(const uint8_t *src, int n, int src_w, int src_h, int chan_order,
                    int rotate180, int resize_mode, int quantize_u8, uint16_t *dst_nhwc8,
                    uint8_t *rotated_or_null, int device);
/* boxes f32[n][A][4] xyxy, scores f32[n][A][nc] (host).  Outputs per frame: max_det entries. */
int irmv_nms(const float *boxes, const float *scores, int n, int anchors, int nc, float score_thr,
             float iou_thr, int max_det, int32_t *num_dets, float *det_boxes, float *det_scores,
             int32_t *det_classes, int32_t *det_index, int device);
/* head tensors (host FP16): box [n][A][64], cls [n][A][16] in anchor order -> decoded boxes and
 * scores (host f32), the decode half of the fused decode+NMS kernel. */
int irmv_decode(const uint16_t *box_nhwc, const uint16_t *cls_nhwc, int n, float *boxes,
                float *scores, int device);

/* ---- PnP ----------------------------------------------------------------------------------- */
int irmv_pnp_create(const double K[9], const double D[5], int device, irmv_pnp **out);
void irmv_pnp_destroy(irmv_pnp *p);
/* img_pts: {LB.x,LB.y, LT.x,LT.y, RT.x,RT.y, RB.x,RB.y} (src/pnp_solver.cpp:41-44). ok=1 solved. */
int irmv_pnp_solve(irmv_pnp *p, const float img_pts[8], double rvec[3], double tvec[3], int *ok);
int irmv_pnp_solve_batch(irmv_pnp *p, const float *img_pts, int n, int on_device, int large_armor,
                         double *rvecs, double *tvecs, uint8_t *ok);
/* Extended output: quaternion (x,y,z,w) as tf2::Matrix3x3::getRotation gives
 * (src/irm_detector.cpp:218-226) and both IPPE solutions' RMSE; any pointer may be NULL. */
int irmv_pnp_solve_batch_ex(irmv_pnp *p, const float *img_pts, int n, int on_device,
                            int large_armor, double *rvecs, double *tvecs, uint8_t *ok,
                            double *quats, double *rvecs2, double *tvecs2, double *rmse2);
/* Optional stage, OFF by default (= reference behaviour: cv::solvePnP(..., SOLVEPNP_IPPE) does not refine,
 * src/pnp_solver.cpp:49-51): max_iters > 0 adds a Levenberg-Marquardt refinement of the returned pose on the pixel
 * reprojection error (the north_star's "IPPE + LM"; oracle cv2.solvePnPRefineLM).  Second solution and RMSE outputs of
 * _ex stay IPPE's. */
int irmv_pnp_set_refine_lm(irmv_pnp *p, int max_iters);
double irmv_pnp_last_device_ms(irmv_pnp *p);
float irmv_pnp_distance_to_center(irmv_pnp *p, float x, float y);

#ifdef __cplusplus
}
#endif
#endif /* IRMV_CABI_H_ */
