// K0: per-stream APE state machine and motion predictor, one thread per stream.
//
// Device restatement of detect_pose.py:467-574 (accept / reset rules),
// detect_pose.py:229-301 (relative motion, 2-deep velocity FIFOs, acceleration)
// and detect_pose.py:303-349 + transform_helper.py:123-259 (constant-acceleration
// extrapolation composed as 4x4 matrices, Euler half-angle of the rotational
// acceleration, float32 tvec of the predicted guess).  It also reproduces what
// cv::solvePnP(useExtrinsicGuess=True) does to the caller's arrays: the result
// is written INTO the guess arrays (dtype preserved), and those arrays may be
// the same objects as prev_transform (detect_pose.py:551,569).
//
// State record (AGT_STREAM_STATE_DOUBLES doubles per stream):
//   [0] has_prev  [1..6] prev pose  [7] has_guess  [8..13] guess pose
//   [14] guess arrays alias prev arrays  [15] guess tvec is float32
//   [16] n_vel  [17..25] rot_vel[0]  [26..28] tran_vel[0]  [29..37] rot_vel[1]  [38..40] tran_vel[1]
//   [41] prev tvec is float32 (prev holds the arrays of a float32 guess)
#include "agt_common.cuh"

namespace {

enum { S_HAS_PREV = 0, S_PREV = 1, S_HAS_GUESS = 7, S_GUESS = 8, S_ALIAS = 14, S_T32 = 15, S_NVEL = 16, S_RV0 = 17,
       S_TV0 = 26, S_RV1 = 29, S_TV1 = 38, S_P32 = 41 };
static_assert(S_HAS_GUESS == AGT_STATE_HAS_GUESS && S_GUESS == AGT_STATE_GUESS, "agt_common.cuh: state record slots");

__device__ inline void mat3_mul(const double* A, const double* B, double* C) {      // C = A B
  for (int r = 0; r < 3; ++r)
    for (int c = 0; c < 3; ++c) C[r * 3 + c] = A[r * 3] * B[c] + A[r * 3 + 1] * B[3 + c] + A[r * 3 + 2] * B[6 + c];
}
__device__ inline void mat3_tmul(const double* A, const double* B, double* C) {     // C = A^T B
  for (int r = 0; r < 3; ++r)
    for (int c = 0; c < 3; ++c) C[r * 3 + c] = A[r] * B[c] + A[3 + r] * B[3 + c] + A[6 + r] * B[6 + c];
}
__device__ inline void mat3_tvec(const double* A, const double* v, double* o) {     // o = A^T v
  for (int r = 0; r < 3; ++r) o[r] = A[r] * v[0] + A[3 + r] * v[1] + A[6 + r] * v[2];
}

__global__ void ape_prepare_kernel(const double* __restrict__ state, double* __restrict__ guess,
                                   uint8_t* __restrict__ use_guess, int batch, int enhance) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= batch) return;
  const double* s = state + (int64_t)i * AGT_STREAM_STATE_DOUBLES;
  bool use = enhance && s[S_HAS_GUESS] != 0.0;              // detect_pose.py:508
  use_guess[i] = use ? 1 : 0;
  for (int k = 0; k < 6; ++k) guess[(int64_t)i * 6 + k] = use ? s[S_GUESS + k] : 0.0;
}

// detect_pose.py:490-574 for one stream: s = its state record, p_in = the pose solvePnP (or the dense refinement)
// returned.  Returns accepted; error is set where the reference would raise ValueError.
__device__ inline bool ape_update_stream(double* s, int n_tags, const double* p_in, bool ok, float err, int enhance, bool& error) {
  error = false;
  double held[6];
  for (int k = 0; k < 6; ++k) held[k] = s[S_PREV + k];      // deepcopy(prev_transform), detect_pose.py:490
  if (n_tags < 2) { s[S_HAS_GUESS] = 0.0; return false; }   // detect_pose.py:494-496,573-574
  const bool fresh = !(enhance && s[S_HAS_GUESS] != 0.0);
  const bool t32 = !fresh && s[S_T32] != 0.0;                // the pose lands in float32 tvec arrays
  double p[6];
  for (int k = 0; k < 6; ++k) p[k] = p_in[k];
  if (!fresh) {
    // solvePnP wrote its result into the guess arrays (dtype preserved)
    if (t32)
      for (int k = 3; k < 6; ++k) p[k] = (double)(float)p[k];
    for (int k = 0; k < 6; ++k) s[S_GUESS + k] = p[k];
    if (s[S_ALIAS] != 0.0)
      for (int k = 0; k < 6; ++k) s[S_PREV + k] = p[k];
  }
  if (!ok) return false;                                     // detect_pose.py:533
  if (!(err < 2.0f)) { s[S_HAS_GUESS] = 0.0; return false; } // detect_pose.py:539,570-572
  if (fresh) {
    for (int k = 0; k < 6; ++k) s[S_GUESS + k] = p[k];       // detect_pose.py:551
    s[S_HAS_GUESS] = 1.0; s[S_ALIAS] = 1.0; s[S_T32] = 0.0;
  } else {
    // get_pose_vel_acc(curr, held_prev)  detect_pose.py:245-301
    double Rp[9], Rcur[9], rv[9], tv[3], dt[3];
    agt_rodrigues(held, Rp);
    agt_rodrigues(p, Rcur);
    // numpy subtracts two float32 tvec arrays in float32 (both are float32 values already: one rounding)
    const bool f32_sub = t32 && s[S_P32] != 0.0;
    for (int k = 0; k < 3; ++k) dt[k] = f32_sub ? (double)__fsub_rn((float)held[3 + k], (float)p[3 + k]) : held[3 + k] - p[3 + k];
    mat3_tvec(Rcur, dt, tv);                                 // R_curr^T (t_prev - t_curr)
    mat3_tmul(Rcur, Rp, rv);                                 // R_curr^T R_prev
    bool zero = false;
    for (int k = 0; k < 9; ++k) zero = zero || rv[k] == 0.0;
    for (int k = 0; k < 3; ++k) zero = zero || tv[k] == 0.0;
    if (zero) {                                              // detect_pose.py:236-237 raises ValueError
      error = true;
      return true;                                           // (the pose passed the gate; the state update is abandoned)
    }
    int nv = (int)s[S_NVEL];
    if (nv >= 2) {                                           // FIFO depth 2: drop the oldest
      for (int k = 0; k < 9; ++k) s[S_RV0 + k] = s[S_RV1 + k];
      for (int k = 0; k < 3; ++k) s[S_TV0 + k] = s[S_TV1 + k];
      nv = 1;
    }
    double* rdst = nv == 0 ? s + S_RV0 : s + S_RV1;
    double* tdst = nv == 0 ? s + S_TV0 : s + S_TV1;
    for (int k = 0; k < 9; ++k) rdst[k] = rv[k];
    for (int k = 0; k < 3; ++k) tdst[k] = tv[k];
    ++nv;
    s[S_NVEL] = (double)nv;
    if (nv > 1) {
      // accelerations, detect_pose.py:291-299 (index 1 = newest)
      const double* rv_new = s + S_RV1; const double* rv_old = s + S_RV0;
      double dtv[3], tacc[3], racc[9];
      for (int k = 0; k < 3; ++k) dtv[k] = s[S_TV0 + k] - s[S_TV1 + k];
      mat3_tvec(rv_new, dtv, tacc);
      mat3_tmul(rv_new, rv_old, racc);
      // apply_vel_acc(held_prev, ...)  detect_pose.py:303-349
      double sy = sqrt(racc[0] * racc[0] + racc[3] * racc[3]);
      double ex, ey, ez;
      if (!(sy < 1e-6)) { ex = atan2(racc[7], racc[8]); ey = atan2(-racc[6], sy); ez = atan2(racc[3], racc[0]); }
      else { ex = atan2(-racc[5], racc[4]); ey = atan2(-racc[6], sy); ez = 0.0; }
      ex *= 0.5; ey *= 0.5; ez *= 0.5;
      double cx = cos(ex), sx = sin(ex), cy = cos(ey), sy2 = sin(ey), cz = cos(ez), sz = sin(ez);
      double Rx[9] = {1, 0, 0, 0, cx, -sx, 0, sx, cx};
      double Ry[9] = {cy, 0, sy2, 0, 1, 0, -sy2, 0, cy};
      double Rz[9] = {cz, -sz, 0, sz, cz, 0, 0, 0, 1};
      double Ryx[9], Ra[9];
      mat3_mul(Ry, Rx, Ryx);
      mat3_mul(Rz, Ryx, Ra);                                 // transform_helper.py:235
      // pred = E(Ra, 0.5 tacc) E(rv, tv) E(Rprev, tprev)    detect_pose.py:334-341
      double R1[9], t1[3], R2[9], t2[3];
      mat3_mul(rv, Rp, R1);
      for (int r = 0; r < 3; ++r) t1[r] = rv[r * 3] * held[3] + rv[r * 3 + 1] * held[4] + rv[r * 3 + 2] * held[5] + tv[r];
      mat3_mul(Ra, R1, R2);
      for (int r = 0; r < 3; ++r) t2[r] = Ra[r * 3] * t1[0] + Ra[r * 3 + 1] * t1[1] + Ra[r * 3 + 2] * t1[2] + 0.5 * tacc[r];
      double rvec[3];
      agt_log_rotation(R2, rvec);                            // cv.Rodrigues(rmat), detect_pose.py:344
      // cv::Rodrigues orthonormalises the matrix by an SVD first, which fails on a non-finite matrix: the vector is zero.  The
      // reference's 4x4 product also makes the rotation non-finite where a translation is (times the next factor's zero row).
      bool fin = true;
      for (int k = 0; k < 9; ++k) fin = fin && isfinite(R2[k]);
      for (int k = 0; k < 3; ++k) fin = fin && isfinite(tacc[k]) && isfinite(tv[k]);
      if (!fin) rvec[0] = rvec[1] = rvec[2] = 0.0;
      for (int k = 0; k < 3; ++k) s[S_GUESS + k] = rvec[k];
      for (int k = 0; k < 3; ++k) s[S_GUESS + 3 + k] = (double)(float)t2[k];   // transform_helper.py:158-159
      s[S_HAS_GUESS] = 1.0; s[S_ALIAS] = 0.0; s[S_T32] = 1.0;
    } else {
      s[S_ALIAS] = 1.0;                                      // guess arrays are now also prev_transform
    }
  }
  for (int k = 0; k < 6; ++k) s[S_PREV + k] = p[k];          // detect_pose.py:569
  s[S_HAS_PREV] = 1.0;
  s[S_P32] = t32 ? 1.0 : 0.0;
  return true;
}

__global__ void ape_update_kernel(double* __restrict__ state, const int32_t* __restrict__ n_tags,
                                  const double* __restrict__ pose, const uint8_t* __restrict__ ok,
                                  const float* __restrict__ err, uint8_t* __restrict__ accepted,
                                  uint8_t* __restrict__ error_flag, int batch, int enhance) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= batch) return;
  bool error;
  const bool acc = ape_update_stream(state + (int64_t)i * AGT_STREAM_STATE_DOUBLES, n_tags[i], pose + (int64_t)i * 6, ok[i] != 0,
                                     err[i], enhance, error);
  if (accepted) accepted[i] = acc ? 1 : 0;
  if (error_flag) error_flag[i] = error ? 1 : 0;
}

// The reference's acceptance test of a solved frame (detect_pose.py:494, 533, 539): at least two tags, solvePnP
// succeeded, mean reprojection error below 2 px.  Used to mask the dense refinement.
__global__ void accept_gate_kernel(const uint8_t* __restrict__ ok, const float* __restrict__ err, const int32_t* __restrict__ n_tags,
                                   uint8_t* __restrict__ gate, int batch) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < batch) gate[i] = ok[i] != 0 && err[i] < 2.0f && n_tags[i] >= 2 ? 1 : 0;
}

// One warp per stream: lane 0 applies the state update with the refined pose where the refinement produced one,
// then the warp hands the frame's corners over to the next LK step (PoseDetector._prev_corners keeps the corners of
// accepted frames only) and publishes the stream's pose.
__global__ void ape_commit_kernel(double* __restrict__ state, const int32_t* __restrict__ n_tags, const double* __restrict__ pose,
                                  const uint8_t* __restrict__ ok, const float* __restrict__ err,
                                  const double* __restrict__ refined_pose, const uint8_t* __restrict__ refined_status,
                                  const float* __restrict__ img, const uint8_t* __restrict__ valid, float* __restrict__ prev_pts,
                                  uint8_t* __restrict__ prev_valid, int n_pts, uint8_t* __restrict__ accepted,
                                  uint8_t* __restrict__ error_flag, double* __restrict__ pose_out, int batch, int enhance) {
  const int i = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (i >= batch) return;
  double* s = state + (int64_t)i * AGT_STREAM_STATE_DOUBLES;
  int acc = 0;
  if (lane == 0) {
    const bool use_refined = refined_pose != nullptr && refined_status != nullptr && refined_status[i] != 0;
    const double* p = use_refined ? refined_pose + (int64_t)i * 6 : pose + (int64_t)i * 6;
    bool error;
    const bool a = ape_update_stream(s, n_tags[i], p, ok[i] != 0, err[i], enhance, error);
    acc = a ? 1 : 0;
    if (accepted) accepted[i] = (uint8_t)acc;
    if (error_flag) error_flag[i] = error ? 1 : 0;
  }
  acc = __shfl_sync(0xffffffffu, acc, 0);
  __syncwarp();
  if (pose_out && lane < 6) pose_out[(int64_t)i * 6 + lane] = s[S_PREV + lane];
  if (prev_pts && prev_valid && img && valid) {
    for (int k = lane; k < 2 * n_pts; k += 32) prev_pts[(int64_t)i * 2 * n_pts + k] = img[(int64_t)i * 2 * n_pts + k];
    for (int k = lane; k < n_pts; k += 32) prev_valid[(int64_t)i * n_pts + k] = acc ? valid[(int64_t)i * n_pts + k] : 0;
  }
}

// where the detector has to look in the next frame of a stream: the image of the object's bounding sphere at the predicted pose
// (the extrinsic guess, detect_pose.py:553-566) or else at the last accepted pose, plus a margin; no pose -> the whole frame
__global__ void track_rects_kernel(const double* __restrict__ state, agt_camera cam, double radius, int margin, int w, int h,
                                   int32_t* __restrict__ rects, int batch) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= batch) return;
  const double* s = state + (int64_t)i * AGT_STREAM_STATE_DOUBLES;
  const double* t = s[S_HAS_GUESS] != 0.0 ? s + S_GUESS + 3 : (s[S_HAS_PREV] != 0.0 ? s + S_PREV + 3 : nullptr);
  int r[4] = {0, 0, 0, 0};                                   // empty rectangle: search the whole frame
  if (t != nullptr && t[2] > 1e-6 && t[0] == t[0] && t[1] == t[1]) {
    double ext[4];
    for (int a = 0; a < 2; ++a) {
      const double c = t[a], f = a == 0 ? cam.fx : cam.fy, pp = a == 0 ? cam.cx : cam.cy;
      const double sb = fmin(radius / sqrt(c * c + t[2] * t[2]), 0.95);
      const double al = atan2(c, t[2]), be = asin(sb);
      ext[2 * a] = f * tan(fmax(al - be, -1.5)) + pp - margin;
      ext[2 * a + 1] = f * tan(fmin(al + be, 1.5)) + pp + margin;
    }
    const int x0 = (int)fmax(floor(ext[0]), 0.0), y0 = (int)fmax(floor(ext[2]), 0.0);
    const int x1 = (int)fmin(ceil(ext[1]) + 1.0, (double)w), y1 = (int)fmin(ceil(ext[3]) + 1.0, (double)h);
    if (x1 > x0 && y1 > y0) { r[0] = x0; r[1] = y0; r[2] = x1; r[3] = y1; }
  }
  reinterpret_cast<int4*>(rects)[i] = make_int4(r[0], r[1], r[2], r[3]);
}

}  // namespace

extern "C" int agt_track_rects(agt_ctx* ctx, const double* d_state, double radius, int margin, int w, int h, int32_t* d_rects, int batch) {
  if (!ctx) return AGT_ERR_INVALID;
  if (batch == 0) return AGT_OK;
  if (!ctx->camera_set) AGT_FAIL(ctx, AGT_ERR_NOT_READY, "agt_track_rects: no camera set");
  if (!d_state || !d_rects || batch < 0 || !(radius > 0.0) || margin < 0 || w < 1 || h < 1 || (reinterpret_cast<uintptr_t>(d_rects) & 15) != 0)
    AGT_FAIL(ctx, AGT_ERR_INVALID, "agt_track_rects: bad arguments (d_rects 16-byte aligned)");
  track_rects_kernel<<<(batch + 127) / 128, 128, 0, ctx->stream>>>(d_state, ctx->cam, radius, margin, w, h, d_rects, batch);
  AGT_LAUNCH_CHECK(ctx);
  return AGT_OK;
}

extern "C" int agt_ape_prepare(agt_ctx* ctx, const double* d_state, double* d_guess, uint8_t* d_use_guess, int batch,
                               int enhance_ape) {
  if (!ctx) return AGT_ERR_INVALID;
  if (batch == 0) return AGT_OK;          // nothing to do (empty tensors may carry null pointers)
  if (!d_state || !d_guess || !d_use_guess || batch < 0) AGT_FAIL(ctx, AGT_ERR_INVALID, "agt_ape_prepare: bad arguments");
  if (batch == 0) return AGT_OK;
  ape_prepare_kernel<<<(batch + 127) / 128, 128, 0, ctx->stream>>>(d_state, d_guess, d_use_guess, batch, enhance_ape);
  AGT_LAUNCH_CHECK(ctx);
  return AGT_OK;
}

extern "C" int agt_ape_update(agt_ctx* ctx, double* d_state, const int32_t* d_n_tags, const double* d_pose,
                              const uint8_t* d_ok, const float* d_err, uint8_t* d_accepted, uint8_t* d_error_flag,
                              int batch, int enhance_ape) {
  if (!ctx) return AGT_ERR_INVALID;
  if (batch == 0) return AGT_OK;          // nothing to do (empty tensors may carry null pointers)
  if (!d_state || !d_n_tags || !d_pose || !d_ok || !d_err || batch < 0)
    AGT_FAIL(ctx, AGT_ERR_INVALID, "agt_ape_update: bad arguments");
  if (batch == 0) return AGT_OK;
  ape_update_kernel<<<(batch + 63) / 64, 64, 0, ctx->stream>>>(d_state, d_n_tags, d_pose, d_ok, d_err, d_accepted,
                                                              d_error_flag, batch, enhance_ape);
  AGT_LAUNCH_CHECK(ctx);
  return AGT_OK;
}

extern "C" int agt_accept_gate(agt_ctx* ctx, const uint8_t* d_ok, const float* d_err, const int32_t* d_n_tags, uint8_t* d_gate, int batch) {
  if (!ctx) return AGT_ERR_INVALID;
  if (batch == 0) return AGT_OK;          // nothing to do (empty tensors may carry null pointers)
  if (!d_ok || !d_err || !d_n_tags || !d_gate || batch < 0) AGT_FAIL(ctx, AGT_ERR_INVALID, "agt_accept_gate: bad arguments");
  accept_gate_kernel<<<(batch + 127) / 128, 128, 0, ctx->stream>>>(d_ok, d_err, d_n_tags, d_gate, batch);
  AGT_LAUNCH_CHECK(ctx);
  return AGT_OK;
}

extern "C" int agt_ape_commit(agt_ctx* ctx, double* d_state, const int32_t* d_n_tags, const double* d_pose, const uint8_t* d_ok,
                              const float* d_err, const double* d_refined_pose, const uint8_t* d_refined_status,
                              const float* d_img_pts, const uint8_t* d_valid, float* d_prev_pts, uint8_t* d_prev_valid, int n_pts,
                              uint8_t* d_accepted, uint8_t* d_error_flag, double* d_pose_out, int batch, int enhance_ape) {
  if (!ctx) return AGT_ERR_INVALID;
  if (batch == 0) return AGT_OK;          // nothing to do (empty tensors may carry null pointers)
  if (!d_state || !d_n_tags || !d_pose || !d_ok || !d_err || batch < 0 || n_pts < 0 || n_pts > AGT_MAX_POINTS)
    AGT_FAIL(ctx, AGT_ERR_INVALID, "agt_ape_commit: bad arguments");
  ape_commit_kernel<<<(batch + 3) / 4, 128, 0, ctx->stream>>>(d_state, d_n_tags, d_pose, d_ok, d_err, d_refined_pose, d_refined_status,
                                                             d_img_pts, d_valid, d_prev_pts, d_prev_valid, n_pts, d_accepted,
                                                             d_error_flag, d_pose_out, batch, enhance_ape);
  AGT_LAUNCH_CHECK(ctx);
  return AGT_OK;
}

