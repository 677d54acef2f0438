/*
 * agt.h - C ABI of the B200-native AprilGroup tracking hot path (libagt.so).
 *
 * The reference (Virtana/accurate-aprilgroup-tracking) has no FFI of its own: its
 * hot path is Python calling OpenCV.  Every entry point below therefore names
 * the reference call site / OpenCV call it stands in for.  A maintainer binds
 * these with ctypes (see INTEGRATION.md); nothing here uses torch or C++ types.
 *
 * Conventions
 *   - every function returns 0 on success or a negative agt_status; it never
 *     throws or aborts.  agt_last_error() returns a message for the last failure.
 *   - per-item failures (a corner lost by LK, a PnP that did not converge) are
 *     reported in status arrays, not as error codes.
 *   - "d_" pointers are device pointers on the context's device, "h_" pointers
 *     are host pointers.  Device entry points are asynchronous on the context's
 *     stream (agt_set_stream); host entry points copy, run and synchronise.
 *   - a pose is 6 doubles: rvec (axis-angle, OpenCV convention) then tvec,
 *     X_cam = R(rvec) X_group + tvec  (detect_pose.py:528).
 *   - a context is bound to one CUDA device and is not re-entrant; use one
 *     context (and one process) per GPU.
 */
#ifndef AGT_H_
#define AGT_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define AGT_VERSION 100
#define AGT_MAX_LEVELS 4
#define AGT_MAX_TAGS 16
#define AGT_MAX_POINTS 64 /* 4 corners x AGT_MAX_TAGS */

typedef enum agt_status {
  AGT_OK = 0,
  AGT_ERR_INVALID = -1,   /* bad argument (maps to ValueError) */
  AGT_ERR_CUDA = -2,      /* CUDA runtime failure (maps to RuntimeError) */
  AGT_ERR_NOT_READY = -3, /* camera / group / model not set */
  AGT_ERR_NO_DEVICE = -4  /* no usable CUDA device: there is no CPU fallback */
} agt_status;

typedef struct agt_ctx agt_ctx;

/* A batch of gray image pyramids resident in device memory.  Level l of frame
 * b starts at data[l] + b*frame_stride[l]; rows are pitch[l] bytes apart.
 * Level 0 is the input frame; levels 1.. are cv::pyrDown chains of it. */
typedef struct agt_pyramid {
  int32_t levels;
  int32_t width[AGT_MAX_LEVELS];
  int32_t height[AGT_MAX_LEVELS];
  int64_t pitch[AGT_MAX_LEVELS];
  int64_t frame_stride[AGT_MAX_LEVELS];
  uint8_t* data[AGT_MAX_LEVELS];
} agt_pyramid;

/* per-refinement status (dense pose refinement) */
enum { AGT_DPR_NONE = 0, AGT_DPR_CONVERGED = 1, AGT_DPR_MAX_EVALS = 2, AGT_DPR_LAMBDA = 3 };

/* ---- lifecycle ----------------------------------------------------------- */
int agt_version(void);
int agt_device_count(void);
int agt_create(int device, agt_ctx** out);
int agt_destroy(agt_ctx* ctx);
const char* agt_last_error(const agt_ctx* ctx); /* ctx may be NULL: last create() error */
/* Run all subsequent device work of this context on `cuda_stream` (a
 * cudaStream_t, e.g. torch.cuda.current_stream().cuda_stream; 0/NULL is the
 * CUDA legacy default stream, which is what torch uses unless told otherwise).
 * A fresh context runs on its own non-blocking stream until this is called. */
int agt_set_stream(agt_ctx* ctx, void* cuda_stream);
int agt_sync(agt_ctx* ctx);
/* number of kernel launches issued by this context since creation */
int64_t agt_launch_count(const agt_ctx* ctx);

/* ---- configuration --------------------------------------------------------- */
/* Camera matrix (row-major 3x3) and 0/4/5 distortion coefficients k1 k2 p1 p2 [k3]
 * - the mtx/dist pair the reference passes to cv.solvePnP / cv.projectPoints
 * (detect_pose.py:509-526, transform_helper.py:106-111). */
int agt_set_camera(agt_ctx* ctx, const double k[9], const double* dist, int ndist);
/* Surface model for dense refinement: samples[S][4] = x,y,z (group frame) and
 * target intensity; sample_tag[S] in [0,n_tags); samples must be tag-major
 * (all samples of tag 0, then tag 1, ...).  pitch = metric sample spacing. */
int agt_set_model(agt_ctx* ctx, const float* h_samples, const uint8_t* h_sample_tag, int n_samples,
                  const float* h_tag_normals, const float* h_tag_centres, int n_tags, double pitch);

/* ---- frame ingest: cv::cvtColor(frame, COLOR_BGR2GRAY) (detect_pose.py:602), bit-exact for 8-bit images ---- */
/* d_bgr[batch][h][src_pitch] interleaved B,G,R -> d_gray[batch][h][dst_pitch] (e.g. level 0 of a pyramid). */
int agt_bgr_to_gray(agt_ctx* ctx, const uint8_t* d_bgr, int w, int h, int64_t src_pitch, int64_t src_stride,
                    uint8_t* d_gray, int64_t dst_pitch, int64_t dst_stride, int batch);

/* ---- frame ingest with lens undistortion: undistort_frame (detect_pose.py:147-183, called by process_frame,
 * detect_pose.py:611-619) followed by BGR2GRAY (detect_pose.py:602), bit-exact for 8-bit frames --------------- */
/* new_K[9] (row-major, [[fx s cx] [0 fy cy] [0 0 1]]) and the crop are what cv.getOptimalNewCameraMatrix returns
 * for width x height frames; the lens model is the one given to agt_set_camera.  Must be called again when the
 * camera or the frame size changes. */
int agt_set_undistort(agt_ctx* ctx, const double* new_K, int width, int height, int roi_x, int roi_y, int roi_w, int roi_h);
/* d_src[batch][h][src_pitch], 1 (gray) or 3 (B,G,R interleaved) channels -> d_gray[batch][roi_h][dst_pitch] =
 * cvtColor(undistort(frame, K, dist, None, new_K)[roi], BGR2GRAY), e.g. straight into level 0 of a roi_w x roi_h
 * pyramid.  cv::undistort arithmetic: float64 maps rounded to 1/32 px, cv::remap's int16 bilinear table,
 * BORDER_CONSTANT 0. */
int agt_undistort_to_gray(agt_ctx* ctx, const uint8_t* d_src, int w, int h, int channels, int64_t src_pitch,
                          int64_t src_stride, uint8_t* d_gray, int64_t dst_pitch, int64_t dst_stride, int batch);
/* One frame from host memory: h_src[h][w][channels] -> h_gray[roi_h][roi_w]. */
int agt_undistort_to_gray_host(agt_ctx* ctx, const uint8_t* h_src, int w, int h, int channels, uint8_t* h_gray);
/* cv::undistort + crop alone, channels kept: d_dst[batch][roi_h][dst_pitch] = undistort(frame, K, dist, None, new_K)[roi] - the frame
 * undistort_frame returns (detect_pose.py:174-181), which the reference goes on to draw on and display. */
int agt_undistort_frames(agt_ctx* ctx, const uint8_t* d_src, int w, int h, int channels, int64_t src_pitch, int64_t src_stride,
                  uint8_t* d_dst, int64_t dst_pitch, int64_t dst_stride, int batch);
/* process_frame (detect_pose.py:611-619) for one host frame with one upload: h_frame[roi_h][roi_w][channels] (may be NULL) as
 * agt_undistort, h_gray[roi_h][roi_w] (may be NULL) as agt_undistort_to_gray. */
int agt_undistort_frame_host(agt_ctx* ctx, const uint8_t* h_src, int w, int h, int channels, uint8_t* h_frame, uint8_t* h_gray);

/* ---- N3 (first step): sub-pixel corner refinement around given (predicted / tracked / detected) corners --------------------
 * cv::cornerSubPix(gray, corners, (win, win), (-1, -1), (COUNT + EPS, max_iters, eps)) per frame of a batch - the corner
 * refinement of OpenCV's ArUco detector, which stands in for the `refine_edges` step of the reference's apriltag detector
 * (detect_pose.py:86-95, :368-371; that library is not vendored).  d_pts / d_out [batch][n_pts][2] float32, d_valid
 * [batch][n_pts] (NULL = all): points that are not valid or lie outside the frame are copied through.  win = 1..7. */
int agt_corner_subpix(agt_ctx* ctx, const uint8_t* d_gray, int w, int h, int64_t pitch, int64_t stride, const float* d_pts,
                      const uint8_t* d_valid, float* d_out, int batch, int n_pts, int win, int max_iters, double eps);
/* One host image, corners refined in place (the OpenCV calling convention). */
int agt_corner_subpix_host(agt_ctx* ctx, const uint8_t* h_gray, int w, int h, float* h_pts, int n_pts, int win, int max_iters,
                           double eps);

/* ---- N3: tag identification (detect_pose.py:368-400: which tag, its corner order, the decision-margin filter) --------------
 * agt_set_tag_family: the family's 36-bit code words (tag36h11: 587; first data cell of the top row = most significant bit).
 * agt_decode_tags: d_quads [batch][n_quads][4][2] float32 in the reference's corner order (transform_helper.py:56-59: bottom-left,
 * top-left, top-right, bottom-right of the printed tag; any cyclic rotation of it is accepted) -> d_id (-1: no tag), d_rotation
 * (the quad's first corner is the tag's corner d_rotation), d_hamming, d_margin (mean distance of the 64 cell means from the
 * threshold: the analogue of apriltag's decision_margin).  Semantics: oracle/tag_oracle.py:decode_np. */
int agt_set_tag_family(agt_ctx* ctx, const uint64_t* h_codes, int n_codes);
int agt_decode_tags(agt_ctx* ctx, const uint8_t* d_gray, int w, int h, int64_t pitch, int64_t stride, const float* d_quads,
                    const uint8_t* d_valid, int32_t* d_id, uint8_t* d_rotation, uint8_t* d_hamming, float* d_margin, int batch,
                    int n_quads, int max_hamming);

/* agt_detect_tags: the detector itself for a batch of gray frames (detect_pose.py:368-371 detector.detect): dark 4-connected
 * components (dark = below darkest + 0.35 x (white - darkest); see agt_set_tag_threshold) -> quadrilateral fit -> agt_corner_subpix (refine_win, 0 = off) -> agt_decode_tags.
 * Per frame up to max_tags tags: d_n_tags [batch] (may exceed max_tags: clamp), d_ids [batch][max_tags], d_corners
 * [batch][max_tags][4][2] in the reference's corner order, d_margin / d_hamming (nullable).  The order of the tags of a frame is
 * not defined.  Pinned to cv2.aruco.ArucoDetector (DICT_APRILTAG_36h11) in tests/: same ids, corners within a pixel. */
int agt_detect_tags(agt_ctx* ctx, const uint8_t* d_gray, int w, int h, int64_t pitch, int64_t stride, int batch, int max_tags,
                    int max_hamming, int refine_win, int32_t* d_n_tags, int32_t* d_ids, float* d_corners, float* d_margin,
                    uint8_t* d_hamming);
int agt_detect_tags_host(agt_ctx* ctx, const uint8_t* h_gray, int w, int h, int max_tags, int max_hamming, int refine_win,
                         int32_t* h_n_tags, int32_t* h_ids, float* h_corners, float* h_margin, uint8_t* h_hamming);
/* What "white" is in the detector's threshold (the reference's apriltag library thresholds adaptively, detect_pose.py:86-95 leaves
 * its defaults): mode 1 = the brightest pixel of the frame's search window, mode 2 = the brightest pixel of the 3 x 3 tiles of
 * 32 x 32 pixels around the pixel (frames lit unevenly), mode 0 (default) = 2 for whole frames, 1 for search windows. */
int agt_set_tag_threshold(agt_ctx* ctx, int mode);
/* The detector on a search window per frame: d_rects [batch][rect_stride >= 4] int32 = x0, y0, x1, y1 in level-0 pixels (clipped to
 * the frame; an empty rectangle = the whole frame; NULL = every frame whole).  Thresholding, components and quads see only the
 * window (a tag cut by the window's edge is dropped like one cut by the frame); results are in frame coordinates.  In a tracking
 * loop the window is the neighbourhood of the predicted object (agt_track_rects): a few percent of a 1080p frame. */
int agt_detect_tags_roi(agt_ctx* ctx, const uint8_t* d_gray, int w, int h, int64_t pitch, int64_t stride, int batch,
                        const int32_t* d_rects, int rect_stride, int max_tags, int max_hamming, int refine_win, int32_t* d_n_tags,
                        int32_t* d_ids, float* d_corners, float* d_margin, uint8_t* d_hamming);
/* The first stage of agt_detect_tags_roi on its own, up to and including the quad emission (same arguments; the detector's
 * max_quads is max(64, 4 max_tags), here 1..4096): per frame d_n_comp = dark components of area >= 48 that were numbered (not
 * clamped: beyond 4096 some are dropped), d_overflow = 1 if the frame took the global-memory union-find, d_n_quads = quads found
 * (not clamped to max_quads), d_quads [batch][max_quads][4][2] (clockwise on the screen, frame coordinates; slot order not
 * defined, slots beyond d_n_quads undefined) and d_quad_win [batch][max_quads], the window agt_detect_tags refines each quad's
 * corners with.  Semantics: oracle/tag_oracle.py:quads_np. */
int agt_tag_quads(agt_ctx* ctx, const uint8_t* d_gray, int w, int h, int64_t pitch, int64_t stride, int batch, const int32_t* d_rects,
                  int rect_stride, int max_quads, int refine_win, int32_t* d_n_comp, uint8_t* d_overflow, int32_t* d_n_quads,
                  float* d_quads, uint8_t* d_quad_win);
/* Search windows from the stream states (see agt_ape_prepare): the image of a sphere of `radius` metres around the group's origin
 * at the predicted pose (the extrinsic guess, detect_pose.py:553-566), else at the last accepted pose, grown by `margin` pixels;
 * streams without a pose get the empty rectangle (= whole frame).  d_rects [batch][4] int32, 16-byte aligned. */
int agt_track_rects(agt_ctx* ctx, const double* d_state, double radius, int margin, int w, int h, int32_t* d_rects, int batch);
/* A0 on the device (detect_pose.py:385-437 _obtain_detections): the output of agt_detect_tags -> the arrays the batched path
 * takes.  Detections with d_det_margin < min_margin are dropped (detect_pose.py:389, the reference's 50; NULL margins keep all);
 * the corners of the tag with id d_group_ids[k] (the group's ids in JSON key order, detect_pose.py:122) go to d_img_pts
 * [batch][n_group][4][2] at position k with d_valid [batch][n_group][4] = 1, everything else is zero; a tag seen twice keeps the
 * detection with the larger margin; d_n_tags [batch] = tags placed; d_n_unknown [batch] (nullable) = kept detections whose id is
 * not in the group (the reference raises KeyError on those, detect_pose.py:408-415: the host wrapper does the same). */
int agt_pack_detections(agt_ctx* ctx, const int32_t* d_n_det, const int32_t* d_det_ids, const float* d_det_corners,
                        const float* d_det_margin, int max_tags, const int32_t* d_group_ids, int n_group, float min_margin,
                        float* d_img_pts, uint8_t* d_valid, int32_t* d_n_tags, int32_t* d_n_unknown, int batch);

/* ---- N4: the overlay after the path, batched (detect_pose.py:441-465 _project_draw_points; draw.py:120-153) --------------
 * For every frame with a non-zero d_frame_mask entry (NULL = all) and every point: (x, y) = np.round(d_pts) and, if
 * 0 <= x < bound_w and 0 <= y < bound_h (the reference tests against 1280 x 720), cv.circle(img, (x, y), radius,
 * (blue, green, red), -1) into d_bgr[batch][h][pitch] (3 interleaved channels) - bit-identical to the cv.circle loop.
 * d_pts [batch][n_pts][2] float64 is what agt_project writes.  The reference uses radius 5 and (0, 0, 255). */
int agt_draw_points(agt_ctx* ctx, uint8_t* d_bgr, int w, int h, int64_t pitch, int64_t stride, const double* d_pts,
                    const uint8_t* d_frame_mask, int batch, int n_pts, int radius, int bound_w, int bound_h, int blue, int green,
                    int red);

/* ---- K1: image pyramid + Scharr (cv::pyrDown / cv::Scharr, bit-exact) ------- */
/* One pyrDown step on a batch: dst is ((w+1)/2) x ((h+1)/2). */
int agt_pyr_down(agt_ctx* ctx, const uint8_t* d_src, int w, int h, int64_t src_pitch, int64_t src_stride,
                 uint8_t* d_dst, int64_t dst_pitch, int64_t dst_stride, int batch);
/* Fill levels 1..levels-1 of every frame from level 0. */
int agt_build_pyramid(agt_ctx* ctx, const agt_pyramid* pyr, int batch);
/* Region-of-interest variants (the three stages only ever read the neighbourhood of the tracked object):
 * _roi fills, per frame, only the part of levels 1.. that lies below its level-0 rectangle
 * d_rects[b*rect_stride + 0..3] = x0,y0,x1,y1 (x multiples of 16; pixels whose 5x5 support chain lies inside
 * the rectangle are bit-identical to the full pyramid, the rest of the level is left untouched);
 * _masked rebuilds the full pyramid of the frames with any non-zero entry in d_mask[b*mask_stride ..]. */
int agt_build_pyramid_roi(agt_ctx* ctx, const agt_pyramid* pyr, const int32_t* d_rects, int rect_stride, int batch);
int agt_build_pyramid_masked(agt_ctx* ctx, const agt_pyramid* pyr, const uint8_t* d_mask, int mask_stride, int batch);
/* Interleaved (dx,dy) int16 Scharr planes, d_dst[b][h][w][2] (the layout
 * cv::buildOpticalFlowPyramid(withDerivatives=true) produces). */
int agt_scharr(agt_ctx* ctx, const uint8_t* d_src, int w, int h, int64_t src_pitch, int64_t src_stride,
               int16_t* d_dst, int batch);

/* ---- K2: pyramidal Lucas-Kanade (cv::calcOpticalFlowPyrLK defaults) --------- */
/* winSize 21x21, pyr->levels levels, criteria (COUNT+EPS, 30, 0.01),
 * minEigThreshold 1e-4, flags 0.  Points are [batch][n_pts][2] float32. */
int agt_lk(agt_ctx* ctx, const agt_pyramid* prev, const agt_pyramid* next, const float* d_prev_pts,
           float* d_next_pts, uint8_t* d_status, float* d_err, int batch, int n_pts);

/* Same, but frames with d_n_tags[b] >= 2 are skipped (status 0, points copied through): in the pipeline tracking
 * only backs up frames in which fewer than two tags were detected. */
int agt_lk_fallback(agt_ctx* ctx, const agt_pyramid* prev, const agt_pyramid* next, const float* d_prev_pts,
                    float* d_next_pts, uint8_t* d_status, float* d_err, const int32_t* d_n_tags, int batch, int n_pts);
/* Tracking on region-of-interest pyramids (agt_build_pyramid_roi): tracking reads only the neighbourhood of the corners,
 * so the pyramid of a new frame need not be built anywhere else.
 * agt_lk_rects: d_rects[b*rect_stride + 0..3] = level-0 rectangle (x0,y0,x1,y1; x multiples of 16) that covers everything
 * tracking the points of frame b (d_valid[b][n_pts] selects them, NULL = all) can read while no corner moves more than
 * max_flow pixels: bounding box of the points + (16 + 2) * 2^(levels-1) + max_flow.
 * agt_lk_roi: agt_lk / agt_lk_fallback (d_n_tags may be NULL) on pyramids built under d_rects_prev / d_rects_next (either
 * may be NULL: that pyramid is complete).  The results are exact by construction: d_left_roi[b][n_pts] flags every corner
 * whose template footprint or search region left the part of a level that is bit-identical to the full pyramid; the
 * caller rebuilds the flagged frames (agt_any_flag + agt_build_pyramid_masked) and calls again with d_mask (NULL = all
 * frames; otherwise only frames with a non-zero entry are tracked and the outputs of the others are left untouched). */
int agt_lk_rects(agt_ctx* ctx, const agt_pyramid* pyr, const float* d_pts, const uint8_t* d_valid, int n_pts, int max_flow,
                 int32_t* d_rects, int rect_stride, int batch);
int agt_lk_roi(agt_ctx* ctx, const agt_pyramid* prev, const agt_pyramid* next, const float* d_prev_pts, float* d_next_pts,
               uint8_t* d_status, float* d_err, const int32_t* d_n_tags, const int32_t* d_rects_prev,
               const int32_t* d_rects_next, int rect_stride, const uint8_t* d_mask, uint8_t* d_left_roi, int batch, int n_pts);
/* Stage-2 integration rule (SURVEY.md 9.2): for every frame with fewer than 2 detected tags, re-admit each
 * tag that was accepted in the previous frame (d_prev_valid) and whose four corners were all tracked
 * (d_status == 1): its tracked corners are copied into d_img_pts and its d_valid entries set.
 * d_n_tags[batch] is recomputed (tags with 4 valid corners); d_tracked_tags[batch] (may be NULL) receives how many
 * tags were re-admitted.  n_pts = 4 * n_tags_total. */
int agt_lk_merge(agt_ctx* ctx, const float* d_tracked_pts, const uint8_t* d_status, const uint8_t* d_prev_valid,
                 float* d_img_pts, uint8_t* d_valid, int32_t* d_n_tags, int32_t* d_tracked_tags, int batch, int n_pts);

/* ---- K3: batched PnP (cv::solvePnP SOLVEPNP_ITERATIVE + reprojection gate) --- */
/* d_obj_pts[n_pts][3] float32 is shared by the batch (group corners, index
 * 4*tag+corner, detect_pose.py:185-227); d_img_pts[batch][n_pts][2] float32;
 * d_valid[batch][n_pts] selects the corners present in a frame (NULL = all).
 * d_guess[batch][6] + d_use_guess[batch] give the extrinsic guess
 * (detect_pose.py:516-526); frames without a guess start from a DLT like
 * cv::solvePnP does (detect_pose.py:508-515).  Outputs: pose[batch][6],
 * ok[batch] (solver success), reproj_err[batch] = mean L2 pixel error
 * (transform_helper.py:98-121), iters[batch] (may be NULL). */
int agt_pnp(agt_ctx* ctx, const float* d_obj_pts, const float* d_img_pts, const uint8_t* d_valid,
            const double* d_guess, const uint8_t* d_use_guess, double* d_pose, uint8_t* d_ok,
            float* d_reproj_err, int32_t* d_iters, int batch, int n_pts);
/* cv::projectPoints: d_out[batch][n_pts][2] float64. */
int agt_project(agt_ctx* ctx, const float* d_obj_pts, const double* d_pose, double* d_out, int batch, int n_pts);

/* The stream pipeline's one-warp-per-frame steps around K3 in ONE launch (a frame-step is a chain of dependent launches):
 * agt_lk_merge (d_tracked_pts NULL: skipped) -> agt_ape_prepare (the guess is read from the state records, detect_pose.py:508)
 * -> agt_pnp -> agt_accept_gate (d_gate, may be NULL; detect_pose.py:494, 533, 539) and d_refine_status[batch] = 0 (may be NULL).
 * d_img_pts / d_valid are merged in place; d_n_tags_in[batch] is read, d_n_tags[batch] written (they may be the same array).
 * Same arithmetic, frame by frame, as the separate calls. */
int agt_streams_front(agt_ctx* ctx, const float* d_obj_pts, const float* d_tracked_pts, const uint8_t* d_lk_status,
                      const uint8_t* d_prev_valid, float* d_img_pts, uint8_t* d_valid, const int32_t* d_n_tags_in, int32_t* d_n_tags,
                      int32_t* d_tracked_tags, const double* d_state, int enhance_ape, double* d_pose, uint8_t* d_ok,
                      float* d_reproj_err, int32_t* d_iters, uint8_t* d_gate, uint8_t* d_refine_status, int batch, int n_pts);

/* ---- K0: per-stream APE state machine + motion predictor --------------------- */
/* State of one camera stream as detect_pose.py:74-78 keeps it (prev_transform,
 * extrinsic_guess, 2-deep velocity FIFOs) plus the aliasing flags needed to
 * reproduce cv::solvePnP's in-place write into the guess arrays. Opaque
 * 64-double record per stream; zero-initialise for a fresh stream. */
#define AGT_STREAM_STATE_DOUBLES 64
/* Before K3: write guess[batch][6]/use_guess[batch] from the states. */
int agt_ape_prepare(agt_ctx* ctx, const double* d_state, double* d_guess, uint8_t* d_use_guess, int batch,
                    int enhance_ape);
/* After K3 (+ optional refinement): apply detect_pose.py:490-574 to each
 * stream. n_tags[batch] = accepted detections in the frame; pose/ok/err from
 * agt_pnp.  accepted[batch] (may be NULL) receives 1 where prev_transform was
 * updated. error_flag[batch] (may be NULL) is set where the reference would
 * raise ValueError (exact zero in a velocity, detect_pose.py:236-237). */
int agt_ape_update(agt_ctx* ctx, double* d_state, const int32_t* d_n_tags, const double* d_pose,
                   const uint8_t* d_ok, const float* d_err, uint8_t* d_accepted, uint8_t* d_error_flag,
                   int batch, int enhance_ape);
/* d_gate[batch] = the reference's acceptance test of a solved frame (detect_pose.py:494, 533, 539): at least two
 * tags, solvePnP succeeded, mean reprojection error below 2 px.  Masks the dense refinement of a stream step. */
int agt_accept_gate(agt_ctx* ctx, const uint8_t* d_ok, const float* d_err, const int32_t* d_n_tags, uint8_t* d_gate, int batch);
/* agt_ape_update for a stream step with dense refinement and LK: where d_refined_status[batch] != 0 the refined
 * pose d_refined_pose[batch][6] replaces the PnP pose before it becomes prev_transform (both may be NULL); then the
 * frame's corners are handed to the next LK step (d_prev_pts = d_img_pts, d_prev_valid = d_valid where the frame was
 * accepted, else 0: PoseDetector keeps the corners of accepted frames only; all four may be NULL) and
 * d_pose_out[batch][6] (may be NULL) receives each stream's prev_transform. */
int agt_ape_commit(agt_ctx* ctx, double* d_state, const int32_t* d_n_tags, const double* d_pose, const uint8_t* d_ok,
                   const float* d_err, const double* d_refined_pose, const uint8_t* d_refined_status,
                   const float* d_img_pts, const uint8_t* d_valid, float* d_prev_pts, uint8_t* d_prev_valid, int n_pts,
                   uint8_t* d_accepted, uint8_t* d_error_flag, double* d_pose_out, int batch, int enhance_ape);

/* ---- K4: dense pose refinement (photometric LM; DodecaPen stage 3) ----------- */
/* d_init[batch][n_hyp][6] -> d_pose[batch][n_hyp][6]; cost = 1/2 sum r^2,
 * n_valid = samples in the final residual, evals = cost/Jacobian evaluations
 * run, status = AGT_DPR_*.  Any output except d_pose may be NULL.  d_mask[batch]
 * (may be NULL) skips frames whose entry is 0: none of their outputs is
 * written.  d_left_roi[batch][n_hyp] (may be NULL) is set
 * to 1 when a sample ever read pixels outside the region of interest predicted
 * from the initial pose (projected bounding sphere + 8 px drift margin). */
int agt_refine(agt_ctx* ctx, const agt_pyramid* pyr, const double* d_init, int n_hyp, const uint8_t* d_mask,
               double* d_pose, float* d_cost, int32_t* d_n_valid, int32_t* d_evals, uint8_t* d_status,
               uint8_t* d_left_roi, int batch);
/* As agt_refine, with K1 fused into K4: only level 0 of `pyr` has to hold the frames.  Each refinement builds the
 * part of levels 1..l it reads (its predicted ROI, grown by the 5x5 support of every pyrDown above it) from
 * level 0 inside the kernel - cv2.pyrDown arithmetic, bit-identical to agt_build_pyramid - and writes it into
 * the pyramid's buffers; everything else in levels >= 1 is left untouched.  Results are identical to
 * agt_build_pyramid + agt_refine unless left_roi is set; such frames must be redone on a full pyramid
 * (agt_build_pyramid_masked + masked agt_refine), exactly as after agt_build_pyramid_roi. */
int agt_refine_fused(agt_ctx* ctx, const agt_pyramid* pyr, const double* d_init, int n_hyp, const uint8_t* d_mask,
                     double* d_pose, float* d_cost, int32_t* d_n_valid, int32_t* d_evals, uint8_t* d_status,
                     uint8_t* d_left_roi, int batch);
/* d_rects[batch][4] (16-byte aligned) = the level-0 rectangle x0,y0,x1,y1 the refinements of each frame can
 * read (predicted ROI of every hypothesis + pyramid halo); feed it to agt_build_pyramid_roi.  A frame whose
 * refinement reports left_roi must be redone on a full pyramid (agt_build_pyramid_masked + masked agt_refine). */
int agt_dpr_rects(agt_ctx* ctx, const agt_pyramid* pyr, const double* d_init, int n_hyp, int32_t* d_rects, int batch);
/* d_out[b] = any(d_flags[b*stride .. b*stride+stride-1]) */
int agt_any_flag(agt_ctx* ctx, const uint8_t* d_flags, int stride, uint8_t* d_out, int batch);
/* Covariance of a refined pose: one evaluation of the refinement's cost function at d_pose[batch][n_hyp][6], the
 * cost function being the one agt_refine fixes from d_init[batch][n_hyp][6] (pyramid level and visible tags decided
 * at the initial pose).  With J the n_valid x 6 Jacobian of the residuals in the refinement's tangent convention -
 * left perturbation R <- exp(w) R, then t <- t + dt; rotation block first (radians), then translation (metres) -
 * and c = 1/2 sum r^2:
 *   d_info[b][h][36] = H = J^T J (row-major, may be NULL),
 *   d_sigma2[b][h]   = s^2 = 2c / (n_valid - 6) (float32, may be NULL; NaN when n_valid <= 6),
 *   d_n_valid[b][h]  = samples in the evaluation (may be NULL),
 *   d_cov[b][h][36]  = Sigma = s^2 H^-1 (row-major, float64),
 *   d_ok[b][h]       = 1, or 0 when n_valid <= 6 or H is not positive definite; Sigma is then NaN.
 * Sigma is the Gauss-Newton covariance of the estimate under independent residuals of equal variance; it is not a
 * bound on the error against the true pose (the estimator's bias is not in it; DESIGN.md section 2).
 * d_mask[batch] (may be NULL) skips frames whose entry is 0: none of their outputs is written.
 * The kernel reads exactly the pixels the refinement's last evaluation read at that pose, so it is valid on a full
 * pyramid, and on a region-of-interest pyramid (agt_build_pyramid_roi) or after agt_refine_fused for every refinement
 * that reported left_roi = 0.  Asynchronous on the context's stream, one launch, graph-capturable. */
int agt_pose_covariance(agt_ctx* ctx, const agt_pyramid* pyr, const double* d_init, const double* d_pose, int n_hyp,
                        const uint8_t* d_mask, double* d_cov, double* d_info, float* d_sigma2, int32_t* d_n_valid,
                        uint8_t* d_ok, int batch);
/* Multi-hypothesis selection: best[b] = argmin_h 2*cost/n_valid (ties -> lowest
 * h); d_best_pose[batch][6] may be NULL. */
int agt_select_best(agt_ctx* ctx, const double* d_pose, const float* d_cost, const int32_t* d_n_valid,
                    int n_hyp, int32_t* d_best, double* d_best_pose, int batch);

/* ---- synthetic input generator (tests / bench only; not part of the path) ---- */
/* Ray-casts the 12-tag dodecahedron of SURVEY.md 8d. d_tag_rt[n_tags][12] =
 * row-major R_k (9) then t_k (3) float64; d_cells[n_tags][100] u8 intensities. */
int agt_render(agt_ctx* ctx, const double* d_pose, const uint32_t* d_seed, uint8_t* d_frames, int w, int h,
               int64_t pitch, int64_t stride, const double* d_tag_rt, const uint8_t* d_cells, int n_tags,
               double inradius, double cell, int noise, int batch);

/* ---- host-buffer entry points (what a ctypes caller with numpy arrays uses) --- */
/* cv.solvePnP(obj, img, K, dist[, rvec, tvec, True], flags=ITERATIVE) for one frame
 * (detect_pose.py:509-526).  pose is in/out when use_guess != 0. */
int agt_solve_pnp_host(agt_ctx* ctx, const float* h_obj, const float* h_img, int n_pts, int use_guess,
                       double h_pose[6], int* ok, float* reproj_err);
int agt_project_host(agt_ctx* ctx, const float* h_obj, int n_pts, const double h_pose[6], double* h_out);
/* cv.calcOpticalFlowPyrLK(prev, next, prevPts, None) on host images. */
int agt_lk_host(agt_ctx* ctx, const uint8_t* h_prev, const uint8_t* h_next, int w, int h, int levels,
                const float* h_prev_pts, int n_pts, float* h_next_pts, uint8_t* h_status, float* h_err);
/* Pyramid of one host image: h_levels[l] receives level l (l >= 1), tightly packed. */
int agt_pyramid_host(agt_ctx* ctx, const uint8_t* h_img, int w, int h, int levels, uint8_t* const* h_levels);
int agt_scharr_host(agt_ctx* ctx, const uint8_t* h_img, int w, int h, int16_t* h_out);
/* cv.cvtColor(frame, cv.COLOR_BGR2GRAY) (detect_pose.py:602) of one host frame h_bgr[h][w][3] -> h_gray[h][w]. */
int agt_bgr_to_gray_host(agt_ctx* ctx, const uint8_t* h_bgr, int w, int h, uint8_t* h_gray);
/* End-to-end batched refinement from HOST frames [batch][h][w] (pinned memory
 * recommended): uploads in chunks overlapped with pyramid construction and
 * refinement, downloads poses.  h_init[batch][n_hyp][6]; outputs as agt_refine
 * plus (n_hyp>1) h_best[batch]. */
/* agt_refine_host uploads, per frame, only the level-0 rectangle its refinement can read (the ROI
 * predicted from the initial pose + pyramid halo) and redoes from the whole frame every frame whose
 * refinement touched pixels outside it, so results are identical to a full upload.  enable = 0
 * always uploads whole frames.  agt_last_h2d_bytes reports what the last call transferred. */
int agt_set_roi_upload(agt_ctx* ctx, int enable);
/* Host frames in PAGEABLE memory (a plain numpy array): `threads` host threads pack each chunk's rectangles into a pinned
 * staging buffer that travels as one copy (default: min(8, hardware threads)); 0 = one 2-D copy per frame.  Frames in pinned,
 * device-mapped memory are read in place by a gather kernel and need neither. */
int agt_set_upload_threads(agt_ctx* ctx, int threads);
int64_t agt_last_h2d_bytes(const agt_ctx* ctx);
int agt_refine_host(agt_ctx* ctx, const uint8_t* h_frames, int w, int h, int levels, int batch,
                    const double* h_init, int n_hyp, double* h_pose, float* h_cost, int32_t* h_n_valid,
                    int32_t* h_evals, uint8_t* h_status, int32_t* h_best);
/* agt_pose_covariance from HOST frames [batch][h][w]: uploads the whole frames, builds their pyramids and evaluates
 * h_init / h_pose [batch][n_hyp][6]; outputs as agt_pose_covariance (h_info, h_sigma2, h_n_valid may be NULL). */
int agt_pose_covariance_host(agt_ctx* ctx, const uint8_t* h_frames, int w, int h, int levels, int batch, const double* h_init,
                             const double* h_pose, int n_hyp, double* h_cov, double* h_info, float* h_sigma2,
                             int32_t* h_n_valid, uint8_t* h_ok);

#ifdef __cplusplus
}
#endif
#endif /* AGT_H_ */
