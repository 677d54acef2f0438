// Shared definitions for libagt.so (sm_100a).  See include/agt.h for the ABI.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "agt.h"

struct agt_camera {
  double fx, fy, cx, cy;
  double k1, k2, p1, p2, k3;
  int has_dist;
};

// frame ingest with undistortion (agt_set_undistort): the new camera matrix, the crop and the stripe height of
// cv::undistort; the distortion itself comes from agt_camera
struct agt_undistort {
  double nfx, nskew, ncx, nfy, ncy;   // new camera matrix (upper triangular)
  double inv_ab, ir0, ir1, ir4;       // stripe-independent entries of its inverse: 1/(fx fy), 1/fx, -s/(fx fy), 1/fy (set on the host)
  int stripe;                         // rows per map stripe: max(1, 4096 / width) of the frame it was set for
  int width, height;                  // frame size it was set for
  int roi_x, roi_y, roi_w, roi_h;     // crop (getOptimalNewCameraMatrix ROI)
};

struct agt_model {
  float4* samples;       // [S] x,y,z,O
  int n_samples;
  int n_tags;
  int tag_begin[AGT_MAX_TAGS + 1];   // sample range per tag (tag-major)
  float normals[AGT_MAX_TAGS][3];
  float centres[AGT_MAX_TAGS][3];
  double pitch;
  double radius;                     // max |sample position|
};

struct agt_ctx {
  int device;
  int sm_count;
  cudaStream_t own_stream;
  cudaStream_t copy_stream;
  cudaStream_t stream;           // where kernels are launched
  cudaEvent_t ev[4];
  int camera_set, model_set, undistort_set;
  agt_camera cam;
  agt_undistort und;
  short* d_remap_tab;            // [1024][4] int16 bilinear weights of cv::remap (device)
  agt_model model;
  int64_t launches;
  int lk_split_max;              // agt_lk of at most this many corners runs a warp per pyramid level (AGT_LK_SPLIT_MAX; 0: never)
  int roi_upload;                // agt_refine_host uploads only the rectangle a refinement can read
  int64_t last_h2d_bytes;        // host->device bytes of the last agt_refine_host call
  int last_redo_frames;          // frames the last agt_refine_host call redid from the full frame
  const uint8_t* host_frames_dev; // device alias of pinned host frames (NULL: pageable memory)
  struct agt_roi_rect* h_rects;  // pinned ROI rectangle lists (double-buffered)
  struct agt_roi_rect* d_rects;
  int rect_capacity;
  // pageable host frames: pinned staging (double-buffered) the upload threads pack ROI rows into, and its device twin
  int upload_threads;            // 0: one 2-D copy per frame
  uint8_t* h_stage[2];
  size_t stage_bytes;
  uint8_t* d_stage;
  cudaEvent_t ev_stage[2];
  struct agt_pack_rect* h_prects;
  struct agt_pack_rect* d_prects;
  int prect_capacity;
  uint64_t* d_tag_codes;         // tag family (36-bit code words) of agt_decode_tags / agt_detect_tags
  int n_tag_codes;
  int tag_threshold;             // agt_set_tag_threshold: 0 auto, 1 one threshold per search window, 2 local white level
  // scratch device memory owned by the context (host entry points)
  void* scratch[8];
  size_t scratch_bytes[8];
  int scratch_in_graph[8];       // the slot's pointer was handed out during a stream capture: never freed before agt_destroy
  void* retired[64];             // outgrown buffers a captured graph may still read
  int n_retired;
  char err[512];
};

extern char g_agt_create_error[512];

#define AGT_FAIL(ctx, code, ...)                                   \
  do {                                                             \
    snprintf((ctx)->err, sizeof((ctx)->err), __VA_ARGS__);         \
    return (code);                                                 \
  } while (0)

#define AGT_CUDA(ctx, call)                                                                   \
  do {                                                                                        \
    cudaError_t e__ = (call);                                                                 \
    if (e__ != cudaSuccess) {                                                                 \
      snprintf((ctx)->err, sizeof((ctx)->err), "%s failed: %s (%s:%d)", #call,                \
               cudaGetErrorString(e__), __FILE__, __LINE__);                                  \
      return AGT_ERR_CUDA;                                                                    \
    }                                                                                         \
  } while (0)

#define AGT_LAUNCH_CHECK(ctx)                                                                 \
  do {                                                                                        \
    (ctx)->launches++;                                                                        \
    cudaError_t e__ = cudaGetLastError();                                                     \
    if (e__ != cudaSuccess) {                                                                 \
      snprintf((ctx)->err, sizeof((ctx)->err), "kernel launch failed: %s (%s:%d)",            \
               cudaGetErrorString(e__), __FILE__, __LINE__);                                  \
      return AGT_ERR_CUDA;                                                                    \
    }                                                                                         \
  } while (0)

// grow-only scratch buffer slot
int agt_scratch(agt_ctx* ctx, int slot, size_t bytes, void** out);

// ---- small device math ------------------------------------------------------
__host__ __device__ __forceinline__ int agt_reflect101(int i, int n) {
  // BORDER_REFLECT_101 for any i (n >= 1)
  if (n == 1) return 0;
  int period = 2 * (n - 1);
  i = i % period;
  if (i < 0) i += period;
  return i < n ? i : period - i;
}

// Rodrigues: rvec -> R (row-major 3x3), double.
__host__ __device__ inline void agt_rodrigues(const double r[3], double R[9]) {
  double th2 = r[0] * r[0] + r[1] * r[1] + r[2] * r[2];
  double th = sqrt(th2);
  if (th < 1e-12) {
    R[0] = 1; R[1] = -r[2]; R[2] = r[1];
    R[3] = r[2]; R[4] = 1; R[5] = -r[0];
    R[6] = -r[1]; R[7] = r[0]; R[8] = 1;
    return;
  }
  double kx = r[0] / th, ky = r[1] / th, kz = r[2] / th;
  double s, c;
  sincos(th, &s, &c);
  double c1 = 1.0 - c;
  R[0] = c + c1 * kx * kx;      R[1] = c1 * kx * ky - s * kz; R[2] = c1 * kx * kz + s * ky;
  R[3] = c1 * ky * kx + s * kz; R[4] = c + c1 * ky * ky;      R[5] = c1 * ky * kz - s * kx;
  R[6] = c1 * kz * kx - s * ky; R[7] = c1 * kz * ky + s * kx; R[8] = c + c1 * kz * kz;
}

// log map: R (row-major) -> rvec, OpenCV convention (angle in [0, pi]).
__host__ __device__ inline void agt_log_rotation(const double R[9], double r[3]) {
  double wx = R[7] - R[5], wy = R[2] - R[6], wz = R[3] - R[1];
  double s = 0.5 * sqrt(wx * wx + wy * wy + wz * wz);
  double c = 0.5 * (R[0] + R[4] + R[8] - 1.0);
  c = c > 1.0 ? 1.0 : (c < -1.0 ? -1.0 : c);
  double th = atan2(s, c);
  if (s > 1e-9) {
    double f = 0.5 * th / s;
    r[0] = wx * f; r[1] = wy * f; r[2] = wz * f;
    return;
  }
  if (c > 0.0) {
    r[0] = 0.5 * wx; r[1] = 0.5 * wy; r[2] = 0.5 * wz;
    return;
  }
  // angle ~ pi: R ~ 2 k k^T - I; take the axis from the largest diagonal entry.
  double k[3];
  int i = (R[0] >= R[4] && R[0] >= R[8]) ? 0 : (R[4] >= R[8] ? 1 : 2);
  int j = (i + 1) % 3, l = (i + 2) % 3;
  k[i] = sqrt(fmax((R[i * 3 + i] + 1.0) * 0.5, 0.0));
  double inv = k[i] > 1e-300 ? 0.25 / k[i] : 0.0;
  k[j] = (R[i * 3 + j] + R[j * 3 + i]) * inv;
  k[l] = (R[i * 3 + l] + R[l * 3 + i]) * inv;
  double sgn = (k[0] * wx + k[1] * wy + k[2] * wz) < 0.0 ? -1.0 : 1.0;
  double nrm = sqrt(k[0] * k[0] + k[1] * k[1] + k[2] * k[2]);
  nrm = nrm > 1e-300 ? nrm : 1e-300;
  r[0] = sgn * th * k[0] / nrm; r[1] = sgn * th * k[1] / nrm; r[2] = sgn * th * k[2] / nrm;
}

// Solve the symmetric positive definite 6x6 system A x = b in place (Cholesky).
// A is full row-major (upper/lower both filled).  Returns false if A is not PD.
__host__ __device__ inline bool agt_chol6_solve(double A[36], double b[6]) {
#pragma unroll
  for (int j = 0; j < 6; ++j) {
    double d = A[j * 6 + j];
    for (int k = 0; k < j; ++k) d -= A[j * 6 + k] * A[j * 6 + k];
    if (!(d > 0.0)) return false;
    d = sqrt(d);
    A[j * 6 + j] = d;
    double inv = 1.0 / d;
    for (int i = j + 1; i < 6; ++i) {
      double v = A[i * 6 + j];
      for (int k = 0; k < j; ++k) v -= A[i * 6 + k] * A[j * 6 + k];
      A[i * 6 + j] = v * inv;
    }
  }
  for (int i = 0; i < 6; ++i) {
    double v = b[i];
    for (int k = 0; k < i; ++k) v -= A[i * 6 + k] * b[k];
    b[i] = v / A[i * 6 + i];
  }
  for (int i = 5; i >= 0; --i) {
    double v = b[i];
    for (int k = i + 1; k < 6; ++k) v -= A[k * 6 + i] * b[k];
    b[i] = v / A[i * 6 + i];
  }
  return true;
}

// 1/sqrt(d) in float64: MUFU.RSQ64H seed (2^-22) + two Newton steps, each three dependent operations deep
__device__ __forceinline__ double agt_rsqrt_newton(double d) {
  double y;
  asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(d));
#pragma unroll
  for (int it = 0; it < 2; ++it) {
    const double e = fma(-(d * y), y, 1.0);
    y = fma(0.5 * y, e, y);
  }
  return y;
}

// 1/d in float64: MUFU.RCP64H seed + two Newton steps (d finite, non-zero, normal)
__device__ __forceinline__ double agt_rcp_newton(double d) {
  double y;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(d));
#pragma unroll
  for (int it = 0; it < 2; ++it) y = fma(fma(-d, y, 1.0), y, y);
  return y;
}

// index of H(p, q), p <= q, in the packed upper triangle stored by rows
__host__ __device__ constexpr int agt_hk(int p, int q) { return p * 6 - p * (p - 1) / 2 + (q - p); }

// Cholesky solve of the SPD system A x = b, A packed as above, everything in registers (all indices are compile-time
// constants).  Right-looking: after the column scale the trailing updates are independent, so the critical path per
// column is one reciprocal square root, one multiplication and one FMA.  L(i, j) overwrites A(j, i).
__device__ __forceinline__ bool agt_chol6_packed(double (&A)[21], double (&b)[6]) {
  double inv[6];
#pragma unroll
  for (int j = 0; j < 6; ++j) {
    const double d = A[agt_hk(j, j)];
    if (!(d > 1e-30 && d < 1e30)) return false;          // not positive definite for our purposes
    const double y = agt_rsqrt_newton(d);
    inv[j] = y;
#pragma unroll
    for (int i = j + 1; i < 6; ++i) A[agt_hk(j, i)] *= y;
#pragma unroll
    for (int k = j + 1; k < 6; ++k)
#pragma unroll
      for (int i = k; i < 6; ++i) A[agt_hk(k, i)] = fma(-A[agt_hk(j, i)], A[agt_hk(j, k)], A[agt_hk(k, i)]);
  }
#pragma unroll
  for (int i = 0; i < 6; ++i) {
    double v = b[i];
#pragma unroll
    for (int k = 0; k < i; ++k) v = fma(-A[agt_hk(k, i)], b[k], v);
    b[i] = v * inv[i];
  }
#pragma unroll
  for (int i = 5; i >= 0; --i) {
    double v = b[i];
#pragma unroll
    for (int k = i + 1; k < 6; ++k) v = fma(-A[agt_hk(i, k)], b[k], v);
    b[i] = v * inv[i];
  }
  return true;
}

__device__ __forceinline__ double agt_warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float agt_warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ long long agt_warp_sum(long long v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// slots of a stream's state record (layout: agt_ape.cu) that other translation units read
constexpr int AGT_STATE_HAS_GUESS = 7, AGT_STATE_GUESS = 8;
