/*
 * opb.h -- C ABI of libopb.so: the B200-native (sm_100a) OpenPose inference hot path.
 *
 * The reference (DeNA/Chainer_Realtime_Multi-Person_Pose_Estimation) is pure Python and has
 * no FFI layer; its drop-in boundary is the Python module `pose_detector`.  This header is the
 * native boundary *underneath* that module: every entry point replaces one block of
 * reference code (cited as file:line relative to the reference tree) and is what a
 * maintainer of the reference would bind with ctypes (see INTEGRATION.md).
 *
 * Conventions
 *   - plain C types only; no torch / numpy types.
 *   - every function returns 0 on success or a negative opb_status; the message is
 *     available from opb_last_error().  The Python wrapper raises on non-zero.
 *   - `loc` arguments: OPB_HOST (pageable or pinned host memory) or OPB_DEVICE (memory on
 *     the context's device).  Output buffers are caller-allocated with an explicit capacity;
 *     the number of valid rows is returned through an int* argument.
 *   - one context per device; calls on one context are serialised on its stream
 *     (opb_set_stream installs a caller-owned cudaStream_t, e.g. torch's current stream).
 *   - there is NO CPU fallback: every compute entry point launches sm_100a kernels.
 */
#ifndef OPB_H_
#define OPB_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define OPB_N_JOINTS 18
#define OPB_N_LIMBS 19
#define OPB_MAX_TAPS 64

typedef enum {
  OPB_OK = 0,
  OPB_ERR_CUDA = -1,          /* CUDA runtime / driver error                                   */
  OPB_ERR_ARG = -2,           /* bad argument                                                  */
  OPB_ERR_STATE = -3,         /* e.g. forward before weights were finalised                    */
  OPB_ERR_CAPACITY = -4,      /* a caller buffer or an internal list overflowed (never silent) */
  OPB_ERR_INDEX = -5,         /* grouping found >=3 matching subsets: the reference raises
                                 IndexError at pose_detector.py:197                            */
  OPB_ERR_UNSUPPORTED = -6
} opb_status;

enum { OPB_HOST = 0, OPB_DEVICE = 1 };
enum { OPB_F32_NCHW = 0, OPB_U8_NHWC_BGR = 1 };          /* opb_forward input formats       */
enum { OPB_PRECISION_FAST = 0, OPB_PRECISION_PARITY = 1, OPB_PRECISION_COMP = 2 };
/* FAST: fp16 operands, fp32 accumulate (map error ~3e-3).  PARITY: split-fp16 (hi+lo, 3 MMAs, two-level accumulation;
 * ~2e-5).  COMP ("compensated"): fp16 main product + 8-bit-float first-order rounding corrections (2 MMAs; ~1e-4),
 * the fastest precision inside north_star's 1e-3 map tolerance. */
enum { OPB_UPSAMPLE_BILINEAR_AC = 0, OPB_UPSAMPLE_BICUBIC = 1 };

/* Constants of entity.py:71-105 (`params`) plus the 21 Gaussian taps of
 * scipy.ndimage.gaussian_filter(sigma=2.5) (pose_detector.py:86), computed by the host in
 * float64 exactly as scipy does, and the capacities of the device-side lists. */
typedef struct opb_params {
  int32_t limbs[OPB_N_LIMBS][2];      /* entity.py:85-105 limbs_point                          */
  double heatmap_peak_thresh;         /* 0.05  entity.py:79                                    */
  double inner_product_thresh;        /* 0.05  entity.py:80                                    */
  double limb_length_ratio;           /* 1.0   entity.py:81                                    */
  double length_penalty_value;        /* 1     entity.py:82                                    */
  double n_subset_limbs_thresh;       /* 3     entity.py:83                                    */
  double subset_score_thresh;         /* 0.2   entity.py:84                                    */
  int32_t n_integ_points;             /* 10    entity.py:77 (only 10 is supported)             */
  int32_t n_integ_points_thresh;      /* 8     entity.py:78                                    */
  int32_t gauss_radius;               /* 10 = int(4.0*2.5+0.5)                                 */
  int32_t reserved0;
  double gauss_taps[OPB_MAX_TAPS];    /* 2*gauss_radius+1 normalised float64 taps              */
  int32_t max_peaks;                  /* per image   (default 8192)                            */
  int32_t max_candidates;             /* per (image, limb) accepted PAF candidates (def 32768) */
  int32_t max_persons;                /* per image subsets alive at any time (default 1024, <= 4096) */
  int32_t reserved1;
} opb_params;

/* Fixed-size per-image result record written by opb_detect_batch (device-resident path) and
 * exchanged between GPUs with one all-gather.  Coordinates are integer peak positions at map
 * resolution so that the host can redo the float64 rescale of pose_detector.py:513-514
 * exactly.  joint id -1 = missing. */
typedef struct opb_person {
  double score;                       /* subsets[:, -2]                                        */
  double count;                       /* subsets[:, -1] (non-integer after a merge, :217)      */
  int32_t peak_id[OPB_N_JOINTS];      /* index into the image's peak table, -1 = none          */
  int32_t x[OPB_N_JOINTS];
  int32_t y[OPB_N_JOINTS];
  int32_t pad[2];
} opb_person;                          /* 16 + 3*72 + 8 = 240 bytes                             */

typedef struct opb_image_header {
  int32_t n_peaks;
  int32_t n_persons;
  int32_t status;                     /* 0 or an opb_status (capacity / index error)           */
  int32_t n_connections;              /* total over the 19 limbs                               */
} opb_image_header;

typedef struct opb_ctx opb_ctx;

/* -- lifetime ---------------------------------------------------------------------------- */
/* replaces PoseDetector.__init__ device selection, pose_detector.py:28-35 */
int opb_create(opb_ctx** out, int device, const opb_params* params);
void opb_destroy(opb_ctx* ctx);
const char* opb_last_error(const opb_ctx* ctx);     /* ctx may be NULL: last create error      */
int opb_set_stream(opb_ctx* ctx, void* cuda_stream); /* cudaStream_t; NULL = context's own     */
int opb_synchronize(opb_ctx* ctx);
int opb_version(void);

/* -- weights: replaces serializers.load_npz(weights_file, model), pose_detector.py:25-26 --- */
/* W is [Cout,Cin,k,k] float32 (Chainer OIHW), b is [Cout]; both host pointers. 92 calls.   */
int opb_load_weights(opb_ctx* ctx, const char* layer, const float* W, const int64_t shape[4],
                     const float* b);
/* repacks to K-major fp16 (and the hi/lo split for OPB_PRECISION_PARITY) and uploads.       */
int opb_finalize_weights(opb_ctx* ctx, int precision_mode);

/* -- CocoPoseNet forward: replaces self.model(x), pose_detector.py:499 / :451
 *    (models/CocoPoseNet.py:132-262).  x: [N,3,H,W] float32 (OPB_F32_NCHW, already
 *    preprocessed as pose_detector.py:426-431) or [N,H,W,3] uint8 BGR (OPB_U8_NHWC_BGR,
 *    /255-0.5 fused into the first conv).  H, W multiples of 8.
 *    paf_out [N,38,H/8,W/8], heat_out [N,19,H/8,W/8] float32.                               */
int opb_forward(opb_ctx* ctx, const void* x, int x_format, int x_loc, int n, int h, int w,
                float* paf_out, float* heat_out, int out_loc);

/* -- upsample: replaces F.resize_images (pose_detector.py:501-502, OPB_UPSAMPLE_BILINEAR_AC:
 *    align-corners bilinear, bit-exact restatement of Chainer's ResizeImages.forward) and one
 *    cv2.resize(INTER_CUBIC) of float maps (pose_detector.py:461-467, OPB_UPSAMPLE_BICUBIC).
 *    in [planes,h,w] -> out [planes,out_h,out_w] float32.  The crop / accumulate / average
 *    steps of detect_precise are inside opb_precise_add_scale.                              */
int opb_upsample(opb_ctx* ctx, int mode, const float* in, int in_loc, int planes, int h, int w,
                 float* out, int out_loc, int out_h, int out_w);

/* -- peaks: replaces compute_peaks_from_heatmaps (CPU branch), pose_detector.py:75-110.
 *    heat [c_plus_1,H,W] float32 (last channel = background, dropped).  peaks_out rows are
 *    (type, x, y, score, id) float64, ordered channel-major then row-major.                 */
int opb_peaks(opb_ctx* ctx, const float* heat, int heat_loc, int c_plus_1, int h, int w,
              double* peaks_out, int peaks_cap, int* n_peaks);

/* -- connections: replaces compute_connections + compute_candidate_connections,
 *    pose_detector.py:135-181.  paf [38,H,W] float32; peaks [n,5] float64 (host).
 *    conn_out rows (id_a, id_b, score) float64, limb after limb; conn_counts[19].           */
int opb_connections(opb_ctx* ctx, const float* paf, int paf_loc, int h, int w, const double* peaks,
                    int n_peaks, double img_len, double* conn_out, int conn_cap, int* conn_counts);

/* -- candidates of ONE limb: replaces compute_candidate_connections, pose_detector.py:135-159.
 *    paf [2,H,W] float32 host; cand_a [n_a,4], cand_b [n_b,4] float64 rows (x, y, score, id).
 *    out rows (id_a, id_b, score) float64, sorted by descending score (stable, :158).          */
int opb_candidates(opb_ctx* ctx, const float* paf, int h, int w, const double* cand_a, int n_a,
                   const double* cand_b, int n_b, double img_len, double* out, int out_cap, int* n_out);

/* -- grouping: replaces grouping_key_points, pose_detector.py:183-250.
 *    subsets_out rows of 20 float64 (18 ids, score, count).                                  */
int opb_group(opb_ctx* ctx, const double* conns, const int* conn_counts, const double* peaks,
              int n_peaks, double* subsets_out, int subsets_cap, int* n_subsets);

/* -- fused device-resident batch path: PoseDetector.__call__ for a batch, pose_detector.py
 *    :493-517 minus the host resize.  imgs [N,H,W,3] uint8 BGR at network-input size.
 *    Runs conv chain -> bilinear upsample to (map_h,map_w) -> peaks -> connections ->
 *    grouping entirely on the device.  headers_out [N], persons_out [N*max_persons]
 *    (host or device per out_loc).  If inject_paf / inject_heat are non-NULL they are
 *    device arrays [N,38,H/8,W/8] / [N,19,H/8,W/8] that REPLACE the network output before
 *    the upsample (the conv chain still runs); used with synthetic 8-person maps because
 *    random weights cannot produce people (SURVEY.md 8d).                                    */
int opb_detect_batch(opb_ctx* ctx, const uint8_t* imgs, int imgs_loc, int n, int h, int w, int map_h,
                     int map_w, double img_len, const float* inject_paf, const float* inject_heat,
                     opb_image_header* headers_out, opb_person* persons_out, int out_loc);

/* -- the post-process half of PoseDetector.__call__ on its own (pose_detector.py:501-512): network outputs
 *    paf_lo [N,38,h8,w8] / heat_lo [N,19,h8,w8] float32 (host or device per maps_loc) -> F.resize_images to
 *    (map_h, map_w) -> peaks -> connections -> grouping, records as in opb_detect_batch.  For callers that run
 *    the network elsewhere, and the entry the no-GPU emulation tests drive (the conv chain cannot be emulated).
 *    With OPB_PAF_LOWRES=1 / OPB_FUSED_PEAKS=1|2 in the environment at opb_create (experimental, also honoured by
 *    opb_detect_batch / opb_detect_image / opb_stream_submit) the PAF line integrals / the peak kernel interpolate
 *    from the low-resolution maps on demand instead of reading materialised full-resolution maps: same results
 *    bit for bit, without the 42 MB per 320x576 image of full-resolution maps going through HBM.            */
int opb_postprocess_batch(opb_ctx* ctx, const float* paf_lo, const float* heat_lo, int maps_loc, int n, int h8,
                          int w8, int map_h, int map_w, double img_len, opb_image_header* headers_out,
                          opb_person* persons_out, int out_loc);

/* -- device-side ingest: replaces cv2.resize(orig_img, (input_w, input_h)) (default INTER_LINEAR on
 *    uint8 BGR, pose_detector.py:493), bit-exact with OpenCV's 8-bit fixed-point path.
 *    src [n,h0,w0,3] -> dst [n,h,w,3] uint8.                                                     */
int opb_resize_linear_u8(opb_ctx* ctx, const uint8_t* src, int src_loc, int n, int h0, int w0,
                         uint8_t* dst, int dst_loc, int h, int w);
/* cv2.resize(orig_img, ..., interpolation=cv2.INTER_CUBIC) on uint8 BGR (detect_precise, pose_detector.py:443):
 * OpenCV's own 8-bit cubic path (int16 Keys taps x 2048, int32 horizontal pass, float32 vertical pass with the
 * fixed-point scalar tail), bit-exact with cv2 when OpenCV does not dispatch to IPP (cv2.ipp.setUseIPP(False), or a
 * build without IPP); IPP's ippiResizeCubic differs from it by 1 LSB in 4-8 % of the pixels.                 */
int opb_resize_cubic_u8(opb_ctx* ctx, const uint8_t* src, int src_loc, int n, int h0, int w0,
                        uint8_t* dst, int dst_loc, int h, int w);
/* PoseDetector.__call__ for ONE frame of arbitrary size (pose_detector.py:484-517): uploads the
 * original frame, resizes it on the device to (in_h, in_w), then runs the same pipeline as
 * opb_detect_batch with n = 1.                                                                  */
int opb_detect_image(opb_ctx* ctx, const uint8_t* img, int img_loc, int orig_h, int orig_w, int in_h,
                     int in_w, int map_h, int map_w, double img_len, opb_image_header* header_out,
                     opb_person* persons_out, int out_loc);

/* -- skeleton overlay: replaces draw_person_pose(orig_img, poses), pose_detector.py:520-553 (the camera loop's
 *    per-frame drawing, camera_pose_demo.py:27).  img [h,w,3] uint8 BGR -> out [h,w,3] = img.copy() with, per person,
 *    the 17 drawn limbs (cv2.line thickness 2; limbs 9 and 13 skipped) and then the joints (cv2.circle radius 3,
 *    filled) in the reference's order and colours, rasterised exactly as OpenCV 4.x does (csrc/overlay.cuh).
 *    poses: host int32 [n_poses,18,3] = poses.round().astype('i') (x, y, visible != 0).  Every drawn joint must lie
 *    inside the image (true for any pose the detector returns); otherwise OPB_ERR_ARG.                           */
int opb_draw_person_pose(opb_ctx* ctx, const uint8_t* img, int img_loc, int h, int w, const int32_t* poses,
                         int n_poses, uint8_t* out, int out_loc);
/* same, taking the persons of image `image_index` of the last detect call straight from the device-resident records
 * (no host round trip of the poses): joint = rint(peak * (sx, sy)) in float64 as :513-514 and :539 compute it
 * (sx = orig_w / map_w, sy = orig_h / map_h; 1, 1 after the precise path).                                        */
int opb_draw_last_result(opb_ctx* ctx, int image_index, const uint8_t* img, int img_loc, int h, int w, double sx,
                         double sy, uint8_t* out, int out_loc);

/* -- streaming mode: the camera loop of camera_pose_demo.py:20-31, pipelined.  Two slots; submit()
 *    enqueues [pinned staging ->] H2D on a copy stream, the device resize (if orig != in), the whole
 *    pipeline and the D2H of the records, and returns without waiting; collect() blocks until that
 *    slot's records are on the host.  Submitting batch i+1 before collecting batch i overlaps its
 *    upload with batch i's kernels.  frames: [n,orig_h,orig_w,3] uint8 BGR, HOST (pinned or pageable) or DEVICE
 *    (used in place; must stay valid until the slot is collected).
 *    inject_* as in opb_detect_batch (device pointers or NULL).                                 */
int opb_stream_submit(opb_ctx* ctx, const uint8_t* frames, int frames_loc, int n, int orig_h, int orig_w,
                      int in_h, int in_w, int map_h, int map_w, double img_len, const float* inject_paf,
                      const float* inject_heat, int slot);
int opb_stream_collect(opb_ctx* ctx, int slot, opb_image_header* headers_out, opb_person* persons_out);
/* Slot 1 runs on a library-owned stream (its kernels fill the tails and launch gaps of slot 0's).  join makes the
 * context's stream (opb_set_stream) wait for every submitted, uncollected batch -- for callers that time or
 * order other work on that stream.                                                              */
int opb_stream_join(opb_ctx* ctx);

/* -- multi-GPU (SURVEY.md 8e: images shard by rank; the reference has no multi-device path, SURVEY 2a) ------------
 * The ONE collective of the path: an ncclAllGather of the fixed-size result records of a streaming slot's batch,
 * [n opb_image_header | n x max_persons opb_person] = opb_record_block_bytes(ctx, n) bytes per rank, straight from
 * the device-resident record block (no host hop), enqueued on the slot's stream behind its pipeline; gathered_dev
 * (device, world x that many bytes) then holds every rank's block in rank order.  opb_stream_collect / opb_stream_join
 * of that slot afterwards also wait for the collective.  NCCL is resolved at run time (dlopen libnccl.so.2, or
 * $OPB_NCCL_LIB) -- the process that calls this already carries it (torch.distributed, or a program linked to NCCL).
 * opb_nccl_unique_id / opb_nccl_comm_init / opb_nccl_comm_destroy wrap ncclGetUniqueId / ncclCommInitRank /
 * ncclCommDestroy for callers without their own NCCL binding (rank 0 creates the 128-byte id and ships it to the
 * other ranks through whatever channel it has; one communicator per process = per GPU).                        */
int opb_nccl_unique_id(uint8_t id_out[128]);
int opb_nccl_comm_init(opb_ctx* ctx, void** nccl_comm_out, int world, int rank, const uint8_t id[128]);
int opb_nccl_comm_destroy(void* nccl_comm);
size_t opb_record_block_bytes(const opb_ctx* ctx, int n);
int opb_allgather_results(opb_ctx* ctx, void* nccl_comm /* ncclComm_t */, int slot, void* gathered_dev);

/* -- face / hand nets (SURVEY 8f#2).  A context whose loaded layers contain "conv6_2_CPM" is a FaceNet /
 *    HandNet context (models/FaceNet.py:10-76, models/HandNet.py; 52 layers, final 1x1 with 71 / 22 channels):
 *    opb_forward then returns only heat_out [n, 71|22, h/8, w/8] and uint8 input is normalised /256 - 0.5
 *    (face_detector.py:32).
 *    opb_keypoints_detect = FaceDetector.__call__ (face_detector.py:28-41) / HandDetector.__call__
 *    (hand_detector.py:28-51) for one BGR crop [img_h,img_w,3]: device cv2-exact resize to net_size^2,
 *    forward, F.resize_images to the crop size, gaussian_filter(sigma 2.5), per-channel maximum.
 *    out [C-1][3] = (x, y, conf), valid [C-1] = conf > thresh (float32 compare).  mirror = 1 reports positions
 *    in the horizontally flipped maps (hand_type "left": the caller passes the already flipped crop,
 *    hand_detector.py:29-30,46-47).  maps_out (host, may be NULL) receives the unsmoothed upsampled maps.
 *    opb_keypoints_from_heatmaps = compute_peaks_from_heatmaps (face_detector.py:55-67) on caller maps
 *    [planes,h,w] (background channel already dropped).                                          */
int opb_keypoints_detect(opb_ctx* ctx, const uint8_t* img, int img_loc, int img_h, int img_w, int net_size,
                         int mirror, double thresh, double* out, int32_t* valid, float* maps_out);
int opb_keypoints_from_heatmaps(opb_ctx* ctx, const float* heat, int heat_loc, int planes, int h, int w,
                                int mirror, double thresh, double* out, int32_t* valid);
/* FaceDetector / HandDetector __call__ for n crops of different sizes in one pass.  imgs: crops packed back to back
 * (crop i = dims[2i] x dims[2i+1] x 3 uint8 BGR at byte offset sum_{j<i} h_j*w_j*3), host or device; mirror[i] as in
 * opb_keypoints_detect.  out [n][C-1][3], valid [n][C-1]; maps_out (host, may be NULL): the unsmoothed upsampled maps
 * of every crop back to back ([C-1][h_i][w_i] each).
 * One upload, one resize launch, one forward and one launch per post-process stage per chunk: the network runs at the
 * next batch size of 1, 2, 4, 8, 16, 32 (the slots past the last crop hold zeros and are not post-processed), and
 * n > 32 runs in chunks of 32 crops, each ending in one copy of the records to the host and one synchronise.
 * Arguments are checked before anything is launched: n < 0, a NULL array or a crop side <= 0 -> OPB_ERR_ARG (the
 * message names the crop); a pose-net context -> OPB_ERR_STATE; n == 0 -> OPB_OK.  opb_keypoints_detect is the
 * n = 1 case of this call.                                                                                        */
int opb_keypoints_detect_batch(opb_ctx* ctx, const uint8_t* imgs, int imgs_loc, int n, const int32_t* dims,
                               const int32_t* mirror, int net_size, double thresh, double* out, int32_t* valid,
                               float* maps_out);

/* device pointers of the last opb_detect_batch outputs/intermediates (valid until the next
 * call with a different shape): 0 paf_lo, 1 heat_lo, 2 pafs (full-res), 3 heatmaps (full-res),
 * 4 headers, 5 persons, 6 peak table ([N,max_peaks] of {int32 type,x,y; float score}),
 * 7 uint8 network input [N][H][W][3] of the last chain (the resized crops of opb_keypoints_detect_batch)       */
void* opb_device_buffer(opb_ctx* ctx, int which);

/* Detail of image `img` of the last opb_detect_batch / opb_precise_finish: the peak table
 * ([n,5] float64 rows type,x,y,score,id), the 19 connection lists and the kept subsets
 * ([P,20] float64), i.e. the reference's all_peaks / all_connections / subsets.  Any output
 * pointer may be NULL.                                                                       */
int opb_get_image_detail(opb_ctx* ctx, int img, double* peaks_out, int peaks_cap, int* n_peaks,
                         double* conn_out, int conn_cap, int* conn_counts, double* subsets_out,
                         int subsets_cap, int* n_subsets);

/* -- multi-scale precise path: replaces detect_precise, pose_detector.py:433-482 -------------
 * begin: allocate/zero the [38|19, orig_h, orig_w] accumulators.
 * add_scale: padded uint8 BGR image [ph,pw,3] (already resized by the host with
 *   cv2.INTER_CUBIC and padded, :443-445) -> forward -> cubic x8 -> crop pad -> cubic to
 *   (orig_h, orig_w) -> accumulate; the last scale also divides by n_scales (:461-470).
 * finish: peaks -> connections -> grouping on the averaged maps (:475-481).                  */
int opb_precise_begin(opb_ctx* ctx, int orig_h, int orig_w);
int opb_precise_add_scale(opb_ctx* ctx, const uint8_t* img, int img_loc, int ph, int pw, int pad_h,
                          int pad_w, int scale_index, int n_scales);
/* same, with pad_image (pose_detector.py:46-55) on the device: img is the resized, UNPADDED frame [h,w,3];
 * the bottom / right margin up to the next multiple of `stride` is filled with pad_value (B,G,R).  */
int opb_precise_add_scale_unpadded(opb_ctx* ctx, const uint8_t* img, int img_loc, int h, int w, int stride,
                                   const uint8_t pad_value[3], int scale_index, int n_scales);
/* same, starting from the ORIGINAL frame [orig_h,orig_w,3]: the per-scale cv2.resize(..., INTER_CUBIC) to (h, w) of
 * :443 also runs on the device (opb_resize_cubic_u8's kernel), so one scale costs one upload of the original frame and
 * no host arithmetic.                                                                                           */
int opb_precise_add_scale_orig(opb_ctx* ctx, const uint8_t* orig, int img_loc, int orig_h, int orig_w, int h, int w,
                               int stride, const uint8_t pad_value[3], int scale_index, int n_scales);
int opb_precise_finish(opb_ctx* ctx, double img_len, opb_image_header* header_out,
                       opb_person* persons_out, int out_loc);
/* copies the full-resolution maps of image 0 of the current post-process workspace
 * (self.pafs / self.heatmaps of the precise path, :469-470) to the caller.                    */
int opb_download_maps(opb_ctx* ctx, float* pafs_out, float* heat_out, int out_loc);

/* -- instrumentation ---------------------------------------------------------------------- */
/* number of kernels launched by this context since creation (bench.py's gpu_launches)      */
int64_t opb_launch_count(const opb_ctx* ctx);
/* Times `reps` launches of one named stage of the cached pipeline of the last
 * opb_detect_batch / opb_forward shape with CUDA events on the context's stream; returns the
 * mean milliseconds per launch in *ms.  stage: "conv7x7" (the Mconv2..5 grouped launch),
 * "conv_chain", "upsample_paf", "peaks", "paf_integral", ...                                 */
int opb_time_stage(opb_ctx* ctx, const char* stage, int reps, float* ms);

/* -- test hooks (tests/ only) ---------------------------------------------------------------
 * single conv layer through the tcgen05 kernel: x [N,H,W,Cin] fp32 host, W [Cout,Cin,k,k],
 * b [Cout] -> y [N,H,W,Cout] fp32 host (activations are converted to fp16 / split-fp16 on the
 * device exactly as in the chain).  relu: bit 0 = ReLU, bit 1 = fuse the 2x2/2 max-pool (y is
 * then [N,H/2,W/2,Cout]).                                                                    */
int opb_test_conv(opb_ctx* ctx, const float* x, int n, int h, int w, int cin, const float* W,
                  const float* b, int cout, int ksize, int relu, int precision_mode, float* y);

#ifdef __cplusplus
}
#endif
#endif /* OPB_H_ */
