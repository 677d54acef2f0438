// Context lifecycle, configuration and the host-buffer entry points of libagt.so.
#include <new>
#include <thread>
#include <vector>

#include <stdlib.h>
#include <chrono>

#include "agt_dpr_plan.cuh"

char g_agt_create_error[512] = "";

namespace {

inline int64_t align_up(int64_t v, int64_t a) { return (v + a - 1) / a * a; }

// Describe a pyramid for `batch` frames packed into one allocation; returns bytes.
int64_t layout_pyramid(agt_pyramid* p, uint8_t* base, int w, int h, int levels, int batch) {
  memset(p, 0, sizeof(*p));
  p->levels = levels;
  int64_t off = 0;
  for (int l = 0; l < levels; ++l) {
    p->width[l] = w; p->height[l] = h;
    p->pitch[l] = align_up(w, 16);
    p->frame_stride[l] = p->pitch[l] * h;
    p->data[l] = base ? base + off : nullptr;
    off += align_up(p->frame_stride[l] * batch, 256);
    w = (w + 1) / 2; h = (h + 1) / 2;
  }
  return off;
}

}  // namespace

// Growable scratch buffers of the host entry points and of agt_refine's job list.  A CUDA graph that captured a launch reading
// a slot holds the slot's pointer: a slot that has been handed out during a stream capture is never freed before
// agt_destroy (growing it retires the old buffer instead), and it cannot grow DURING a capture (that would need a
// synchronising allocation): run the sequence once eagerly at its final size first.
int agt_scratch(agt_ctx* ctx, int slot, size_t bytes, void** out) {
  if (bytes == 0) bytes = 16;
  cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
  if (cudaStreamIsCapturing(ctx->stream, &cap) != cudaSuccess) { cudaGetLastError(); cap = cudaStreamCaptureStatusNone; }
  const bool capturing = cap == cudaStreamCaptureStatusActive;
  if (ctx->scratch_bytes[slot] < bytes) {
    if (capturing)
      AGT_FAIL(ctx, AGT_ERR_NOT_READY, "scratch slot %d would have to grow (%zu -> %zu bytes) during a stream capture: run the call once "
               "outside the capture at this size first", slot, ctx->scratch_bytes[slot], bytes);
    if (ctx->scratch[slot]) {
      if (ctx->scratch_in_graph[slot]) {
        if (ctx->n_retired >= (int)(sizeof(ctx->retired) / sizeof(ctx->retired[0])))
          AGT_FAIL(ctx, AGT_ERR_NOT_READY, "too many scratch buffers kept alive for captured graphs; destroy the context and its graphs");
        ctx->retired[ctx->n_retired++] = ctx->scratch[slot];      // a captured graph may still read it
      } else {
        AGT_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        AGT_CUDA(ctx, cudaFree(ctx->scratch[slot]));
      }
      ctx->scratch[slot] = nullptr; ctx->scratch_bytes[slot] = 0; ctx->scratch_in_graph[slot] = 0;
    }
    AGT_CUDA(ctx, cudaMalloc(&ctx->scratch[slot], bytes));
    ctx->scratch_bytes[slot] = bytes;
  }
  if (capturing) ctx->scratch_in_graph[slot] = 1;
  *out = ctx->scratch[slot];
  return AGT_OK;
}

extern "C" int agt_version(void) { return AGT_VERSION; }

extern "C" int agt_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
  return n;
}

extern "C" const char* agt_last_error(const agt_ctx* ctx) { return ctx ? ctx->err : g_agt_create_error; }

extern "C" int agt_create(int device, agt_ctx** out) {
  if (!out) { snprintf(g_agt_create_error, sizeof(g_agt_create_error), "agt_create: out is NULL"); return AGT_ERR_INVALID; }
  *out = nullptr;
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n == 0) {
    cudaGetLastError();
    snprintf(g_agt_create_error, sizeof(g_agt_create_error),
             "agt_create: no CUDA device available (%s); this library has no CPU fallback",
             e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0");
    return AGT_ERR_NO_DEVICE;
  }
  if (device < 0 || device >= n) {
    snprintf(g_agt_create_error, sizeof(g_agt_create_error), "agt_create: device %d out of range (0..%d)", device, n - 1);
    return AGT_ERR_INVALID;
  }
  agt_ctx* ctx = new (std::nothrow) agt_ctx();
  if (!ctx) { snprintf(g_agt_create_error, sizeof(g_agt_create_error), "agt_create: out of host memory"); return AGT_ERR_INVALID; }
  memset(ctx, 0, sizeof(*ctx));
  ctx->device = device;
  cudaDeviceProp prop;
  if ((e = cudaSetDevice(device)) != cudaSuccess || (e = cudaGetDeviceProperties(&prop, device)) != cudaSuccess ||
      (e = cudaStreamCreateWithFlags(&ctx->own_stream, cudaStreamNonBlocking)) != cudaSuccess ||
      (e = cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking)) != cudaSuccess) {
    snprintf(g_agt_create_error, sizeof(g_agt_create_error), "agt_create: %s", cudaGetErrorString(e));
    delete ctx;
    return AGT_ERR_CUDA;
  }
  if (prop.major < 10) {
    snprintf(g_agt_create_error, sizeof(g_agt_create_error),
             "agt_create: device %d is sm_%d%d; libagt.so is built for sm_100a only", device, prop.major, prop.minor);
    cudaStreamDestroy(ctx->own_stream); cudaStreamDestroy(ctx->copy_stream);
    delete ctx;
    return AGT_ERR_NO_DEVICE;
  }
  for (int i = 0; i < 4; ++i) cudaEventCreateWithFlags(&ctx->ev[i], cudaEventDisableTiming);
  ctx->sm_count = prop.multiProcessorCount;
  ctx->stream = ctx->own_stream;
  ctx->roi_upload = 1;
  {
    // LK of a small batch (a frame-step of the stream pipeline) is a wait for the slowest corner: a warp per pyramid level
    // (lk_levels_kernel) halves that latency; large batches are throughput-bound and keep one warp per corner.  A machine-full
    // of corners in the level-parallel layout = 4 x 8 CTAs of four warps per SM.
    const char* e = getenv("AGT_LK_SPLIT_MAX");
    ctx->lk_split_max = e ? atoi(e) : 8 * ctx->sm_count;
  }
  {
    unsigned hc = std::thread::hardware_concurrency();
    ctx->upload_threads = hc == 0 ? 4 : (hc < 8 ? (int)hc : 8);
  }
  *out = ctx;
  return AGT_OK;
}

extern "C" int agt_destroy(agt_ctx* ctx) {
  if (!ctx) return AGT_ERR_INVALID;
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  cudaStreamSynchronize(ctx->copy_stream);
  for (int i = 0; i < 8; ++i) if (ctx->scratch[i]) cudaFree(ctx->scratch[i]);
  for (int i = 0; i < ctx->n_retired; ++i) cudaFree(ctx->retired[i]);
  if (ctx->model.samples) cudaFree(ctx->model.samples);
  if (ctx->d_remap_tab) cudaFree(ctx->d_remap_tab);
  if (ctx->d_tag_codes) cudaFree(ctx->d_tag_codes);
  if (ctx->h_rects) cudaFreeHost(ctx->h_rects);
  for (int k = 0; k < 2; ++k) { if (ctx->h_stage[k]) cudaFreeHost(ctx->h_stage[k]); if (ctx->ev_stage[k]) cudaEventDestroy(ctx->ev_stage[k]); }
  for (int i = 0; i < 4; ++i) if (ctx->ev[i]) cudaEventDestroy(ctx->ev[i]);
  cudaStreamDestroy(ctx->own_stream);
  cudaStreamDestroy(ctx->copy_stream);
  delete ctx;
  return AGT_OK;
}

extern "C" int agt_set_stream(agt_ctx* ctx, void* cuda_stream) {
  if (!ctx) return AGT_ERR_INVALID;
  ctx->stream = reinterpret_cast<cudaStream_t>(cuda_stream);   // 0 = the legacy default stream
  return AGT_OK;
}

extern "C" int agt_sync(agt_ctx* ctx) {
  if (!ctx) return AGT_ERR_INVALID;
  AGT_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return AGT_OK;
}

extern "C" int64_t agt_launch_count(const agt_ctx* ctx) { return ctx ? ctx->launches : -1; }

extern "C" int agt_set_camera(agt_ctx* ctx, const double k[9], const double* dist, int ndist) {
  if (!ctx) return AGT_ERR_INVALID;
  if (!k) AGT_FAIL(ctx, AGT_ERR_INVALID, "agt_set_camera: K is NULL");
  if (ndist != 0 && ndist != 4 && ndist != 5) AGT_FAIL(ctx, AGT_ERR_INVALID, "agt_set_camera: ndist must be 0, 4 or 5 (got %d)", ndist);
  if (ndist && !dist) AGT_FAIL(ctx, AGT_ERR_INVALID, "agt_set_camera: dist is NULL");
  if (!(k[0] > 0.0) || !(k[4] > 0.0)) AGT_FAIL(ctx, AGT_ERR_INVALID, "agt_set_camera: focal lengths must be positive");
  agt_camera c;
  memset(&c, 0, sizeof(c));
  c.fx = k[0]; c.fy = k[4]; c.cx = k[2]; c.cy = k[5];
  if (ndist) {
    c.k1 = dist[0]; c.k2 = dist[1]; c.p1 = dist[2]; c.p2 = dist[3]; c.k3 = ndist == 5 ? dist[4] : 0.0;
    c.has_dist = (c.k1 != 0.0 || c.k2 != 0.0 || c.p1 != 0.0 || c.p2 != 0.0 || c.k3 != 0.0);
  }
  ctx->cam = c;
  ctx->camera_set = 1;
  return AGT_OK;
}

extern "C" int agt_set_model(agt_ctx* ctx, const float* h_samples, const uint8_t* h_sample_tag, int n_samples,
                             const float* h_tag_normals, const float* h_tag_centres, int n_tags, double pitch) {
  if (!ctx) return AGT_ERR_INVALID;
  if (!h_samples || !h_sample_tag || !h_tag_normals || !h_tag_centres || n_samples < 1 || n_tags < 1 || n_tags > AGT_MAX_TAGS ||
      !(pitch > 0.0))
    AGT_FAIL(ctx, AGT_ERR_INVALID, "agt_set_model: bad arguments (n_samples=%d n_tags=%d)", n_samples, n_tags);
  agt_model m;
  memset(&m, 0, sizeof(m));
  int tag = 0;
  m.tag_begin[0] = 0;
  for (int i = 0; i < n_samples; ++i) {
    int t = h_sample_tag[i];
    if (t >= n_tags || t < tag) AGT_FAIL(ctx, AGT_ERR_INVALID, "agt_set_model: samples must be tag-major with tags < n_tags (sample %d)", i);
    while (tag < t) m.tag_begin[++tag] = i;
  }
  while (tag < n_tags) m.tag_begin[++tag] = n_samples;
  for (int k = 0; k < n_tags; ++k)
    for (int i = 0; i < 3; ++i) { m.normals[k][i] = h_tag_normals[k * 3 + i]; m.centres[k][i] = h_tag_centres[k * 3 + i]; }
  m.n_samples = n_samples; m.n_tags = n_tags; m.pitch = pitch;
  m.radius = 0.0;                                  // bounding sphere of the surface samples (about the group origin)
  for (int i = 0; i < n_samples; ++i) {
    const float* q = h_samples + 4 * (size_t)i;
    double r = sqrt((double)q[0] * q[0] + (double)q[1] * q[1] + (double)q[2] * q[2]);
    if (r > m.radius) m.radius = r;
  }
  AGT_CUDA(ctx, cudaSetDevice(ctx->device));
  if (ctx->model.samples) { AGT_CUDA(ctx, cudaStreamSynchronize(ctx->stream)); cudaFree(ctx->model.samples); ctx->model.samples = nullptr; }
  AGT_CUDA(ctx, cudaMalloc(&m.samples, sizeof(float4) * (size_t)n_samples));
  AGT_CUDA(ctx, cudaMemcpy(m.samples, h_samples, sizeof(float4) * (size_t)n_samples, cudaMemcpyHostToDevice));
  ctx->model = m;
  ctx->model_set = 1;
  return AGT_OK;
}

// ---------------------------------------------------------------------------------------
// host-buffer entry points
// ---------------------------------------------------------------------------------------
extern "C" int agt_solve_pnp_host(agt_ctx* ctx, const float* h_obj, const float* h_img, int n_pts, int use_guess,
                                  double h_pose[6], int* ok, float* reproj_err) {
  if (!ctx) return AGT_ERR_INVALID;
  if (!h_obj || !h_img || !h_pose || n_pts < 1 || n_pts > AGT_MAX_POINTS)
    AGT_FAIL(ctx, AGT_ERR_INVALID, "agt_solve_pnp_host: bad arguments (n_pts=%d, max %d)", n_pts, AGT_MAX_POINTS);
  AGT_CUDA(ctx, cudaSetDevice(ctx->device));
  uint8_t* d;
  size_t o_obj = 0, o_img = o_obj + 768, o_guess = o_img + 512, o_pose = o_guess + 64, o_err = o_pose + 64, o_ok = o_err + 16,
         o_ug = o_ok + 16, total = o_ug + 16;
  int rc = agt_scratch(ctx, 7, total, reinterpret_cast<void**>(&d));
  if (rc) return rc;
  cudaStream_t st = ctx->stream;
  uint8_t ug = use_guess ? 1 : 0;
  AGT_CUDA(ctx, cudaMemcpyAsync(d + o_obj, h_obj, sizeof(float) * 3 * n_pts, cudaMemcpyHostToDevice, st));
  AGT_CUDA(ctx, cudaMemcpyAsync(d + o_img, h_img, sizeof(float) * 2 * n_pts, cudaMemcpyHostToDevice, st));
  AGT_CUDA(ctx, cudaMemcpyAsync(d + o_guess, h_pose, sizeof(double) * 6, cudaMemcpyHostToDevice, st));
  AGT_CUDA(ctx, cudaMemcpyAsync(d + o_ug, &ug, 1, cudaMemcpyHostToDevice, st));
  rc = agt_pnp(ctx, reinterpret_cast<float*>(d + o_obj), reinterpret_cast<float*>(d + o_img), nullptr,
               reinterpret_cast<double*>(d + o_guess), d + o_ug, reinterpret_cast<double*>(d + o_pose), d + o_ok,
               reinterpret_cast<float*>(d + o_err), nullptr, 1, n_pts);
  if (rc) return rc;
  uint8_t okb = 0;
  float e = 0.f;
  AGT_CUDA(ctx, cudaMemcpyAsync(h_pose, d + o_pose, sizeof(double) * 6, cudaMemcpyDeviceToHost, st));
  AGT_CUDA(ctx, cudaMemcpyAsync(&okb, d + o_ok, 1, cudaMemcpyDeviceToHost, st));
  AGT_CUDA(ctx, cudaMemcpyAsync(&e, d + o_err, sizeof(float), cudaMemcpyDeviceToHost, st));
  AGT_CUDA(ctx, cudaStreamSynchronize(st));
  if (ok) *ok = okb;
  if (reproj_err) *reproj_err = e;
  return AGT_OK;
}

extern "C" int agt_project_host(agt_ctx* ctx, const float* h_obj, int n_pts, const double h_pose[6], double* h_out) {
  if (!ctx) return AGT_ERR_INVALID;
  if (!h_obj || !h_pose || !h_out || n_pts < 1) AGT_FAIL(ctx, AGT_ERR_INVALID, "agt_project_host: bad arguments");
  AGT_CUDA(ctx, cudaSetDevice(ctx->device));
  uint8_t* d;
  size_t o_obj = 0, o_pose = align_up(sizeof(float) * 3 * n_pts, 64), o_out = o_pose + 64, total = o_out + sizeof(double) * 2 * n_pts;
  int rc = agt_scratch(ctx, 7, total, reinterpret_cast<void**>(&d));
  if (rc) return rc;
  cudaStream_t st = ctx->stream;
  AGT_CUDA(ctx, cudaMemcpyAsync(d + o_obj, h_obj, sizeof(float) * 3 * n_pts, cudaMemcpyHostToDevice, st));
  AGT_CUDA(ctx, cudaMemcpyAsync(d + o_pose, h_pose, sizeof(double) * 6, cudaMemcpyHostToDevice, st));
  rc = agt_project(ctx, reinterpret_cast<float*>(d + o_obj), reinterpret_cast<double*>(d + o_pose),
                   reinterpret_cast<double*>(d + o_out), 1, n_pts);
  if (rc) return rc;
  AGT_CUDA(ctx, cudaMemcpyAsync(h_out, d + o_out, sizeof(double) * 2 * n_pts, cudaMemcpyDeviceToHost, st));
  AGT_CUDA(ctx, cudaStreamSynchronize(st));
  return AGT_OK;
}

// upload a tightly packed host image into level 0 of a (batch 1) pyramid
static int upload_level0(agt_ctx* ctx, const agt_pyramid& p, const uint8_t* h_img, cudaStream_t st) {
  AGT_CUDA(ctx, cudaMemcpy2DAsync(p.data[0], (size_t)p.pitch[0], h_img, (size_t)p.width[0], (size_t)p.width[0],
                                  (size_t)p.height[0], cudaMemcpyHostToDevice, st));
  return AGT_OK;
}

extern "C" int agt_pyramid_host(agt_ctx* ctx, const uint8_t* h_img, int w, int h, int levels, uint8_t* const* h_levels) {
  if (!ctx) return AGT_ERR_INVALID;
  if (!h_img || !h_levels || w < 1 || h < 1 || levels < 1 || levels > AGT_MAX_LEVELS)
    AGT_FAIL(ctx, AGT_ERR_INVALID, "agt_pyramid_host: bad arguments");
  AGT_CUDA(ctx, cudaSetDevice(ctx->device));
  agt_pyramid p;
  int64_t bytes = layout_pyramid(&p, nullptr, w, h, levels, 1);
  uint8_t* d;
  int rc = agt_scratch(ctx, 0, (size_t)bytes, reinterpret_cast<void**>(&d));
  if (rc) return rc;
  layout_pyramid(&p, d, w, h, levels, 1);
  cudaStream_t st = ctx->stream;
  if ((rc = upload_level0(ctx, p, h_img, st))) return rc;
  if ((rc = agt_build_pyramid(ctx, &p, 1))) return rc;
  for (int l = 1; l < levels; ++l)
    if (h_levels[l])
      AGT_CUDA(ctx, cudaMemcpy2DAsync(h_levels[l], (size_t)p.width[l], p.data[l], (size_t)p.pitch[l], (size_t)p.width[l],
                                      (size_t)p.height[l], cudaMemcpyDeviceToHost, st));
  AGT_CUDA(ctx, cudaStreamSynchronize(st));
  return AGT_OK;
}

extern "C" int agt_bgr_to_gray_host(agt_ctx* ctx, const uint8_t* h_bgr, int w, int h, uint8_t* h_gray) {
  if (!ctx) return AGT_ERR_INVALID;
  if (!h_bgr || !h_gray || w < 1 || h < 1) AGT_FAIL(ctx, AGT_ERR_INVALID, "agt_bgr_to_gray_host: bad arguments");
  AGT_CUDA(ctx, cudaSetDevice(ctx->device));
  const size_t in_bytes = (size_t)w * h * 3, out_bytes = (size_t)w * h;
  uint8_t *din, *dout;
  int rc;
  if ((rc = agt_scratch(ctx, 0, in_bytes, reinterpret_cast<void**>(&din)))) return rc;
  if ((rc = agt_scratch(ctx, 1, out_bytes, reinterpret_cast<void**>(&dout)))) return rc;
  cudaStream_t st = ctx->stream;
  AGT_CUDA(ctx, cudaMemcpyAsync(din, h_bgr, in_bytes, cudaMemcpyHostToDevice, st));
  if ((rc = agt_bgr_to_gray(ctx, din, w, h, (int64_t)w * 3, (int64_t)in_bytes, dout, w, (int64_t)out_bytes, 1))) return rc;
  AGT_CUDA(ctx, cudaMemcpyAsync(h_gray, dout, out_bytes, cudaMemcpyDeviceToHost, st));
  AGT_CUDA(ctx, cudaStreamSynchronize(st));
  return AGT_OK;
}

extern "C" int agt_scharr_host(agt_ctx* ctx, const uint8_t* h_img, int w, int h, int16_t* h_out) {
  if (!ctx) return AGT_ERR_INVALID;
  if (!h_img || !h_out || w < 1 || h < 1) AGT_FAIL(ctx, AGT_ERR_INVALID, "agt_scharr_host: bad arguments");
  AGT_CUDA(ctx, cudaSetDevice(ctx->device));
  agt_pyramid p;
  int64_t bytes = layout_pyramid(&p, nullptr, w, h, 1, 1);
  uint8_t *d, *dout;
  int rc = agt_scratch(ctx, 0, (size_t)bytes, reinterpret_cast<void**>(&d));
  if (rc) return rc;
  if ((rc = agt_scratch(ctx, 1, sizeof(int16_t) * 2 * (size_t)w * h, reinterpret_cast<void**>(&dout)))) return rc;
  layout_pyramid(&p, d, w, h, 1, 1);
  cudaStream_t st = ctx->stream;
  if ((rc = upload_level0(ctx, p, h_img, st))) return rc;
  if ((rc = agt_scharr(ctx, p.data[0], w, h, p.pitch[0], p.frame_stride[0], reinterpret_cast<int16_t*>(dout), 1))) return rc;
  AGT_CUDA(ctx, cudaMemcpyAsync(h_out, dout, sizeof(int16_t) * 2 * (size_t)w * h, cudaMemcpyDeviceToHost, st));
  AGT_CUDA(ctx, cudaStreamSynchronize(st));
  return AGT_OK;
}

extern "C" int agt_lk_host(agt_ctx* ctx, const uint8_t* h_prev, const uint8_t* h_next, int w, int h, int levels,
                           const float* h_prev_pts, int n_pts, float* h_next_pts, uint8_t* h_status, float* h_err) {
  if (!ctx) return AGT_ERR_INVALID;
  if (!h_prev || !h_next || !h_prev_pts || !h_next_pts || !h_status || !h_err || w < 1 || h < 1 || levels < 1 ||
      levels > AGT_MAX_LEVELS || n_pts < 0)
    AGT_FAIL(ctx, AGT_ERR_INVALID, "agt_lk_host: bad arguments");
  if (n_pts == 0) return AGT_OK;
  AGT_CUDA(ctx, cudaSetDevice(ctx->device));
  // cv::calcOpticalFlowPyrLK lowers maxLevel until the top level is larger than the window
  agt_pyramid pa, pb;
  int64_t bytes = layout_pyramid(&pa, nullptr, w, h, levels, 1);
  uint8_t *da, *db, *dp;
  int rc;
  if ((rc = agt_scratch(ctx, 0, (size_t)bytes, reinterpret_cast<void**>(&da)))) return rc;
  if ((rc = agt_scratch(ctx, 1, (size_t)bytes, reinterpret_cast<void**>(&db)))) return rc;
  size_t o_prev = 0, o_next = align_up(sizeof(float) * 2 * n_pts, 64), o_err = o_next * 2, o_st = o_err + align_up(sizeof(float) * n_pts, 64),
         total = o_st + align_up(n_pts, 64);
  if ((rc = agt_scratch(ctx, 2, total, reinterpret_cast<void**>(&dp)))) return rc;
  layout_pyramid(&pa, da, w, h, levels, 1);
  layout_pyramid(&pb, db, w, h, levels, 1);
  cudaStream_t st = ctx->stream;
  if ((rc = upload_level0(ctx, pa, h_prev, st))) return rc;
  if ((rc = upload_level0(ctx, pb, h_next, st))) return rc;
  AGT_CUDA(ctx, cudaMemcpyAsync(dp + o_prev, h_prev_pts, sizeof(float) * 2 * n_pts, cudaMemcpyHostToDevice, st));
  if ((rc = agt_build_pyramid(ctx, &pa, 1))) return rc;
  if ((rc = agt_build_pyramid(ctx, &pb, 1))) return rc;
  if ((rc = agt_lk(ctx, &pa, &pb, reinterpret_cast<float*>(dp + o_prev), reinterpret_cast<float*>(dp + o_next), dp + o_st,
                   reinterpret_cast<float*>(dp + o_err), 1, n_pts)))
    return rc;
  AGT_CUDA(ctx, cudaMemcpyAsync(h_next_pts, dp + o_next, sizeof(float) * 2 * n_pts, cudaMemcpyDeviceToHost, st));
  AGT_CUDA(ctx, cudaMemcpyAsync(h_status, dp + o_st, n_pts, cudaMemcpyDeviceToHost, st));
  AGT_CUDA(ctx, cudaMemcpyAsync(h_err, dp + o_err, sizeof(float) * n_pts, cudaMemcpyDeviceToHost, st));
  AGT_CUDA(ctx, cudaStreamSynchronize(st));
  return AGT_OK;
}

// One launch copies the ROI rectangle of every frame of a chunk straight out of pinned (device-mapped) host
// memory: 4096 cudaMemcpy2DAsync calls cost ~7 us of driver time each, a gather kernel costs one launch and
// keeps thousands of 16-byte PCIe reads in flight.  rect = (x0, y0, x1, y1, host frame index), x0/x1 % 16 == 0.
struct agt_roi_rect { int x0, y0, x1, y1, src; };

__global__ void __launch_bounds__(256)
roi_gather_kernel(const uint8_t* __restrict__ host_frames, int w, int h, const agt_roi_rect* __restrict__ rects,
                  uint8_t* __restrict__ dst, int64_t dst_pitch, int64_t dst_stride, int n_rects) {
  // a small persistent grid: the CTAs mostly wait on PCIe reads, so they must not fill the SMs' thread
  // slots - the pyramid / refinement kernels of the previous chunk run next to them
  for (int ri = blockIdx.x; ri < n_rects; ri += gridDim.x) {
  const agt_roi_rect r = rects[ri];
  const int cw = (r.x1 - r.x0) >> 4, rows = r.y1 - r.y0;
  if (cw <= 0 || rows <= 0) continue;
  const uint8_t* src = host_frames + (int64_t)r.src * w * h + (int64_t)r.y0 * w + r.x0;
  uint8_t* out = dst + (int64_t)ri * dst_stride + (int64_t)r.y0 * dst_pitch + r.x0;
  // a warp per row, four rows of it in flight: every row is one contiguous run of 16-byte reads, i.e. the fewest
  // 128-byte lines on the bus (host memory is fetched in whole lines: a rectangle padded to 128 B costs the same
  // time as the 16 B aligned one, scripts/gather_probe.cu)
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  for (int y = wid; y < rows; y += 32)
    for (int c0 = 0; c0 < cw; c0 += 32) {
      const int c = c0 + lane;
      uint4 v[4];
#pragma unroll
      for (int k = 0; k < 4; ++k)
        if (y + 8 * k < rows && c < cw) v[k] = *reinterpret_cast<const uint4*>(src + (int64_t)(y + 8 * k) * w + 16 * c);
#pragma unroll
      for (int k = 0; k < 4; ++k)
        if (y + 8 * k < rows && c < cw) *reinterpret_cast<uint4*>(out + (int64_t)(y + 8 * k) * dst_pitch + 16 * c) = v[k];
    }
  }
}

// Pageable host frames (a plain numpy array): the copy engine cannot read them, and one 2-D copy per frame goes through the
// driver's own staging at ~7 us of CPU time each.  Instead a few host threads pack the ROI rows of a chunk into a pinned
// staging buffer (double-buffered), one cudaMemcpyAsync moves the packed chunk, and this kernel puts the rows where the
// refinement reads them.  rect = (x0, y0, x1, y1) with x % 16 == 0, off = byte offset of the rectangle in the packed buffer.
struct agt_pack_rect { int x0, y0, x1, y1; long long off; };

__global__ void __launch_bounds__(256)
roi_scatter_kernel(const uint8_t* __restrict__ packed, const agt_pack_rect* __restrict__ rects, uint8_t* __restrict__ dst,
                   int64_t dst_pitch, int64_t dst_stride, int n_rects) {
  for (int ri = blockIdx.x; ri < n_rects; ri += gridDim.x) {
    const agt_pack_rect r = rects[ri];
    const int cw = (r.x1 - r.x0) >> 4, rows = r.y1 - r.y0;
    if (cw <= 0 || rows <= 0) continue;
    const uint4* src = reinterpret_cast<const uint4*>(packed + r.off);
    uint8_t* out = dst + (int64_t)ri * dst_stride + (int64_t)r.y0 * dst_pitch + r.x0;
    for (int i = threadIdx.x; i < cw * rows; i += blockDim.x) {
      const int y = i / cw, c = i - y * cw;
      *reinterpret_cast<uint4*>(out + (int64_t)y * dst_pitch + 16 * c) = src[i];
    }
  }
}

static void pack_rows(const uint8_t* h_frames, int w, int h, const int* src_frame, const agt_pack_rect* rects, int i0, int i1, uint8_t* stage) {
  for (int i = i0; i < i1; ++i) {
    const agt_pack_rect& r = rects[i];
    const size_t rw = (size_t)(r.x1 - r.x0);
    const uint8_t* src = h_frames + (int64_t)src_frame[i] * w * h + (int64_t)r.y0 * w + r.x0;
    uint8_t* dst = stage + r.off;
    for (int y = r.y0; y < r.y1; ++y, src += w, dst += rw) memcpy(dst, src, rw);
  }
}

extern "C" int agt_set_upload_threads(agt_ctx* ctx, int threads) {
  if (!ctx) return AGT_ERR_INVALID;
  if (threads < 0 || threads > 64) AGT_FAIL(ctx, AGT_ERR_INVALID, "agt_set_upload_threads: 0 (one 2-D copy per frame) .. 64");
  ctx->upload_threads = threads;
  return AGT_OK;
}

extern "C" int agt_set_roi_upload(agt_ctx* ctx, int enable) {
  if (!ctx) return AGT_ERR_INVALID;
  ctx->roi_upload = enable ? 1 : 0;
  return AGT_OK;
}

extern "C" int64_t agt_last_h2d_bytes(const agt_ctx* ctx) { return ctx ? ctx->last_h2d_bytes : -1; }

// scratch slots of agt_refine_host (slot 5 holds the job records of refine_impl in agt_dpr.cu)
constexpr int SLOT_CHUNK0 = 0, SLOT_CHUNK1 = 1, SLOT_JOBS = 2, SLOT_REDO_JOBS = 3, SLOT_RECTS = 4, SLOT_STAGE = 6;

// The per-job arrays of one refinement pass (init and pose: 6 doubles per job; left: the refinement read outside the
// rectangle its frame was given).
struct agt_jobs { double *init, *pose; float* cost; int32_t *n_valid, *evals; uint8_t *status, *left; };

// Lay the arrays of `jobs` jobs out back to back from `base` (nullptr: size only); returns their bytes.
static size_t layout_jobs(agt_jobs* a, uint8_t* base, int64_t jobs) {
  size_t off = 0;
  auto next = [&](size_t per_job) { uint8_t* p = base ? base + off : nullptr; off += align_up(per_job * jobs, 256); return p; };
  a->init = reinterpret_cast<double*>(next(sizeof(double) * 6));
  a->pose = reinterpret_cast<double*>(next(sizeof(double) * 6));
  a->cost = reinterpret_cast<float*>(next(sizeof(float)));
  a->n_valid = reinterpret_cast<int32_t*>(next(sizeof(int32_t)));
  a->evals = reinterpret_cast<int32_t*>(next(sizeof(int32_t)));
  a->status = next(1);
  a->left = next(1);
  return off;
}

// Grow `n` page-locked host buffers of `*bytes` each to at least `need` bytes.  They are kept across calls: page-locking
// memory in every call would add its cost to every call.
static int grow_pinned(agt_ctx* ctx, uint8_t** bufs, int n, size_t* bytes, size_t need) {
  if (*bytes >= need) return AGT_OK;
  for (int k = 0; k < n; ++k) { if (bufs[k]) cudaFreeHost(bufs[k]); bufs[k] = nullptr; }
  *bytes = 0;
  for (int k = 0; k < n; ++k) AGT_CUDA(ctx, cudaMallocHost(reinterpret_cast<void**>(&bufs[k]), need));
  *bytes = need;
  return AGT_OK;
}

static int64_t rect_area(const agt_roi_rect& r) { return (int64_t)(r.x1 - r.x0) * (r.y1 - r.y0); }

// ROI pass: only each frame's rectangle reaches the device, and the refinement builds the part of its pyramid level it
// reads itself (K1 fused into K4).  WHOLE (ROI upload off) and REDO (the frames whose ROI refinement left its rectangle):
// whole frames, full pyramid, plain refinement - the result then cannot depend on any ROI prediction.
enum pass_kind { PASS_ROI, PASS_WHOLE, PASS_REDO };

struct refine_pass_desc {
  pass_kind kind;
  const uint8_t* frames;             // host frames, w x h bytes each
  const uint8_t* frames_dev;         // their device alias (pinned, device-mapped memory) or nullptr
  const double* init;                // host initial poses [frame][n_hyp][6] the ROI pass derives the rectangles from
  int w, h, levels, n_hyp, chunk;
  std::vector<agt_roi_rect> rects;   // per frame of the pass: the level-0 rectangle to upload (empty: none) and its host frame
};

// How the frames of a pass reach the chunk buffers:
//   GATHER  one roi_gather_kernel launch per chunk reads the rectangles out of pinned, device-mapped frames
//   STAGED  host threads pack a chunk's rectangles of pageable frames into pinned staging, one copy, one roi_scatter_kernel
//   WHOLE   one copy per chunk of contiguous whole frames
//   COPIES  one cudaMemcpy2DAsync per rectangle
enum upload_path { UPLOAD_GATHER, UPLOAD_STAGED, UPLOAD_WHOLE, UPLOAD_COPIES };

// One pass of chunked, double-buffered refinement: the H2D of chunk c+1 on the copy stream overlaps the refinement of
// chunk c.  Jobs of chunk c are contiguous in J: [b0*n_hyp, (b0+nb)*n_hyp).
static int refine_pass(agt_ctx* ctx, refine_pass_desc& d, const agt_jobs& J, uint8_t* const buf[2]) {
  cudaStream_t st = ctx->stream, cp = ctx->copy_stream;
  const int count = (int)d.rects.size(), w = d.w, h = d.h;
  // The ROI pass computes its rectangles chunk by chunk, right before the chunk's upload: the CPU work of chunk c+1 then
  // runs while chunk c is copied and refined.  STAGED sizes its staging from all of them, so it computes them up front.
  agt_pyramid one;
  layout_pyramid(&one, nullptr, w, h, d.levels, 1);
  int filled = d.kind == PASS_ROI ? 0 : count;
  auto fill_rects = [&](int end) {
    for (int32_t q[4]; filled < end; ++filled) {
      agt_dpr_rect_l0(ctx->cam, ctx->model.pitch, ctx->model.radius, d.init + (int64_t)filled * d.n_hyp * 6, d.n_hyp, one.width,
                      one.height, one.levels, q);
      d.rects[(size_t)filled] = {q[0], q[1], q[2], q[3], filled};
    }
  };
  // the upload path of this pass (the kernels move 16-byte row pieces; WHOLE needs level 0 at pitch w), and what it
  // needs, set up here and nowhere else
  const bool roi16 = d.kind == PASS_ROI && (w & 15) == 0;
  upload_path path = d.kind == PASS_WHOLE && (w & 15) == 0 ? UPLOAD_WHOLE : UPLOAD_COPIES;
  if (roi16 && d.frames_dev && (reinterpret_cast<uintptr_t>(d.frames_dev) & 15) == 0) path = UPLOAD_GATHER;
  if (roi16 && !d.frames_dev && ctx->upload_threads > 0) path = UPLOAD_STAGED;
  int rc;
  void* d_rects = nullptr;
  uint8_t* d_stage = nullptr;
  if (path == UPLOAD_GATHER || path == UPLOAD_STAGED) {
    // one pinned list slot per frame of the pass, so the CPU never overwrites a list whose asynchronous upload is pending
    const size_t list_bytes = (path == UPLOAD_GATHER ? sizeof(agt_roi_rect) : sizeof(agt_pack_rect)) * (size_t)count;
    if ((rc = grow_pinned(ctx, &ctx->h_rects, 1, &ctx->rect_bytes, list_bytes))) return rc;
    if ((rc = agt_scratch(ctx, SLOT_RECTS, list_bytes, &d_rects))) return rc;
  }
  if (path == UPLOAD_STAGED) {
    // staging: 2 x the largest chunk's rectangles, on the host and on the device
    fill_rects(count);
    int64_t need = 0;
    for (int b0 = 0; b0 < count; b0 += d.chunk) {
      int64_t sum = 0;
      for (int i = b0; i < count && i < b0 + d.chunk; ++i) sum += rect_area(d.rects[(size_t)i]);
      need = sum > need ? sum : need;
    }
    if ((rc = grow_pinned(ctx, ctx->h_stage, 2, &ctx->stage_bytes, (size_t)align_up(need + 256, 4096)))) return rc;
    if ((rc = agt_scratch(ctx, SLOT_STAGE, 2 * ctx->stage_bytes, reinterpret_cast<void**>(&d_stage)))) return rc;
    for (int k = 0; k < 2; ++k)
      if (!ctx->ev_stage[k]) AGT_CUDA(ctx, cudaEventCreateWithFlags(&ctx->ev_stage[k], cudaEventDisableTiming));
  }
  for (int c = 0, b0 = 0; b0 < count; ++c, b0 += d.chunk) {
    const int nb = count - b0 < d.chunk ? count - b0 : d.chunk, s = c & 1;
    const agt_roi_rect* r = d.rects.data() + b0;
    agt_pyramid p;
    layout_pyramid(&p, buf[s], w, h, d.levels, d.chunk);
    if (c >= 2) AGT_CUDA(ctx, cudaStreamWaitEvent(cp, ctx->ev[s], 0));       // compute on this buffer finished
    fill_rects(b0 + nb);
    int64_t bytes = 0;
    for (int i = 0; i < nb; ++i) bytes += rect_area(r[i]);
    if (path == UPLOAD_GATHER) {
      agt_roi_rect* hr = reinterpret_cast<agt_roi_rect*>(ctx->h_rects) + b0;
      agt_roi_rect* drc = static_cast<agt_roi_rect*>(d_rects) + b0;
      memcpy(hr, r, sizeof(agt_roi_rect) * nb);
      AGT_CUDA(ctx, cudaMemcpyAsync(drc, hr, sizeof(agt_roi_rect) * nb, cudaMemcpyHostToDevice, cp));
      // 64 CTAs: enough 16-byte reads in flight to fill PCIe, few enough to leave the SMs to the compute stream
      // (measured 32 / 64 / 128 / 256 CTAs x chunk 128..1024 frames: profiles/r01_e2e_sweep.log)
      roi_gather_kernel<<<nb < 64 ? nb : 64, 256, 0, cp>>>(d.frames_dev, w, h, drc, p.data[0], p.pitch[0], p.frame_stride[0], nb);
      AGT_LAUNCH_CHECK(ctx);
    } else if (path == UPLOAD_STAGED) {
      agt_pack_rect* hr = reinterpret_cast<agt_pack_rect*>(ctx->h_rects) + b0;
      std::vector<int> src_frame((size_t)nb);
      long long off = 0;
      for (int i = 0; i < nb; ++i) {
        src_frame[(size_t)i] = r[i].src;
        hr[i] = {r[i].x0, r[i].y0, r[i].x1, r[i].y1, off};
        off += rect_area(r[i]);
      }
      // the staging buffer of this parity was last read by the copy of chunk c-2
      if (c >= 2) AGT_CUDA(ctx, cudaEventSynchronize(ctx->ev_stage[s]));
      const int nt = ctx->upload_threads < nb ? ctx->upload_threads : nb;
      auto pack = [&](int t) {
        pack_rows(d.frames, w, h, src_frame.data(), hr, (int)((int64_t)nb * t / nt), (int)((int64_t)nb * (t + 1) / nt), ctx->h_stage[s]);
      };
      std::vector<std::thread> pool;
      int t = 1;
      try {
        for (; t < nt; ++t) pool.emplace_back(pack, t);
      } catch (const std::exception&) {}        // slice t found no thread: this thread packs t.. itself (the same bytes)
      pack(0);
      for (int u = t; u < nt; ++u) pack(u);
      for (auto& th : pool) th.join();
      uint8_t* dpk = d_stage + (size_t)s * ctx->stage_bytes;
      agt_pack_rect* drc = static_cast<agt_pack_rect*>(d_rects) + b0;
      AGT_CUDA(ctx, cudaMemcpyAsync(dpk, ctx->h_stage[s], (size_t)off, cudaMemcpyHostToDevice, cp));
      AGT_CUDA(ctx, cudaEventRecord(ctx->ev_stage[s], cp));
      AGT_CUDA(ctx, cudaMemcpyAsync(drc, hr, sizeof(agt_pack_rect) * nb, cudaMemcpyHostToDevice, cp));
      roi_scatter_kernel<<<nb < 296 ? nb : 296, 256, 0, cp>>>(dpk, drc, p.data[0], p.pitch[0], p.frame_stride[0], nb);
      AGT_LAUNCH_CHECK(ctx);
    } else if (path == UPLOAD_WHOLE) {
      AGT_CUDA(ctx, cudaMemcpyAsync(p.data[0], d.frames + (int64_t)b0 * w * h, (size_t)nb * w * h, cudaMemcpyHostToDevice, cp));
    } else {
      for (int i = 0; i < nb; ++i) {
        if (rect_area(r[i]) == 0) continue;
        const agt_roi_rect& q = r[i];
        AGT_CUDA(ctx, cudaMemcpy2DAsync(p.data[0] + (int64_t)i * p.frame_stride[0] + (int64_t)q.y0 * p.pitch[0] + q.x0, (size_t)p.pitch[0],
                                        d.frames + (int64_t)q.src * w * h + (int64_t)q.y0 * w + q.x0, (size_t)w,
                                        (size_t)(q.x1 - q.x0), (size_t)(q.y1 - q.y0), cudaMemcpyHostToDevice, cp));
      }
    }
    ctx->last_h2d_bytes += bytes;
    AGT_CUDA(ctx, cudaEventRecord(ctx->ev[2], cp));
    AGT_CUDA(ctx, cudaStreamWaitEvent(st, ctx->ev[2], 0));
    if (d.kind != PASS_ROI && (rc = agt_build_pyramid(ctx, &p, nb))) return rc;
    const int64_t j0 = (int64_t)b0 * d.n_hyp;
    if ((rc = (d.kind == PASS_ROI ? agt_refine_fused : agt_refine)(ctx, &p, J.init + j0 * 6, d.n_hyp, nullptr, J.pose + j0 * 6,
                                                                   J.cost + j0, J.n_valid + j0, J.evals + j0, J.status + j0,
                                                                   J.left + j0, nb)))
      return rc;
    AGT_CUDA(ctx, cudaEventRecord(ctx->ev[s], st));
  }
  return AGT_OK;
}

extern "C" int agt_refine_host(agt_ctx* ctx, const uint8_t* h_frames, int w, int h, int levels, int batch,
                               const double* h_init, int n_hyp, double* h_pose, float* h_cost, int32_t* h_n_valid,
                               int32_t* h_evals, uint8_t* h_status, int32_t* h_best) try {
  if (!ctx) return AGT_ERR_INVALID;
  if (!ctx->camera_set || !ctx->model_set) AGT_FAIL(ctx, AGT_ERR_NOT_READY, "agt_refine_host: camera and surface model must be set");
  if (!h_frames || !h_init || !h_pose || w < 1 || h < 1 || levels < 1 || levels > AGT_MAX_LEVELS || batch < 0 || n_hyp < 1)
    AGT_FAIL(ctx, AGT_ERR_INVALID, "agt_refine_host: bad arguments");
  ctx->last_h2d_bytes = 0;
  if (batch == 0) return AGT_OK;
  AGT_CUDA(ctx, cudaSetDevice(ctx->device));
  const bool trace = getenv("AGT_TRACE") != nullptr;      // debug aid: phase timestamps on stderr
  auto t_start = std::chrono::steady_clock::now();
  auto since = [&]() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_start).count(); };
  agt_pyramid one;
  int64_t per_frame = layout_pyramid(&one, nullptr, w, h, levels, 1);
  // chunks of up to 1024 frames (<= 3 GiB per buffer): large enough that one refinement launch fills the GPU
  int chunk = (int)((3LL << 30) / per_frame);
  if (chunk > 1024) chunk = 1024;
  if (chunk < 1) chunk = 1;
  if (chunk > batch) chunk = batch;
  int64_t chunk_bytes = layout_pyramid(&one, nullptr, w, h, levels, chunk);
  uint8_t* buf[2];
  int rc;
  if ((rc = agt_scratch(ctx, SLOT_CHUNK0, (size_t)chunk_bytes, reinterpret_cast<void**>(&buf[0])))) return rc;
  if ((rc = agt_scratch(ctx, SLOT_CHUNK1, (size_t)chunk_bytes, reinterpret_cast<void**>(&buf[1])))) return rc;
  const int64_t jobs = (int64_t)batch * n_hyp;
  agt_jobs J;
  const size_t jobs_bytes = layout_jobs(&J, nullptr, jobs);
  uint8_t* dr;
  if ((rc = agt_scratch(ctx, SLOT_JOBS, jobs_bytes + align_up(sizeof(int32_t) * batch, 256), reinterpret_cast<void**>(&dr)))) return rc;
  layout_jobs(&J, dr, jobs);
  int32_t* d_best = reinterpret_cast<int32_t*>(dr + jobs_bytes);
  cudaStream_t st = ctx->stream, cp = ctx->copy_stream;
  AGT_CUDA(ctx, cudaMemcpyAsync(J.init, h_init, sizeof(double) * 6 * jobs, cudaMemcpyHostToDevice, st));
  ctx->last_h2d_bytes += (int64_t)sizeof(double) * 6 * jobs;
  // the copy stream must not overwrite a buffer an earlier call on `st` may still read
  AGT_CUDA(ctx, cudaEventRecord(ctx->ev[3], st));
  AGT_CUDA(ctx, cudaStreamWaitEvent(cp, ctx->ev[3], 0));
  const int roi = ctx->roi_upload && !ctx->cam.has_dist;
  refine_pass_desc d{roi ? PASS_ROI : PASS_WHOLE, h_frames, nullptr, h_init, w, h, levels, n_hyp, chunk,
                     std::vector<agt_roi_rect>((size_t)batch)};
  if (roi) {
    cudaPointerAttributes attr;
    if (cudaPointerGetAttributes(&attr, h_frames) == cudaSuccess && attr.type == cudaMemoryTypeHost && attr.devicePointer)
      d.frames_dev = static_cast<const uint8_t*>(attr.devicePointer);     // pinned + mapped: the gather kernel reads them
    else
      cudaGetLastError();                                                  // pageable
  } else {
    for (int f = 0; f < batch; ++f) d.rects[(size_t)f] = {0, 0, w, h, f};
  }
  if ((rc = refine_pass(ctx, d, J, buf))) return rc;
  if (trace) fprintf(stderr, "[agt] refine_host: first pass enqueued at %.3f ms (chunk %d, roi %d, gather %d)\n", since(), chunk, roi,
                     d.frames_dev != nullptr);
  if (roi) {
    // frames whose refinement read pixels outside the uploaded rectangle are redone from the whole frame,
    // so the result never depends on the ROI prediction
    std::vector<uint8_t> left((size_t)jobs);
    AGT_CUDA(ctx, cudaMemcpyAsync(left.data(), J.left, (size_t)jobs, cudaMemcpyDeviceToHost, st));
    AGT_CUDA(ctx, cudaStreamSynchronize(st));
    std::vector<int> ids;
    for (int f = 0; f < batch; ++f) {
      bool any = false;
      for (int k = 0; k < n_hyp; ++k) any = any || left[(size_t)f * n_hyp + k];
      if (any) ids.push_back(f);
    }
    const int n_redo = (int)ids.size();
    if (trace) fprintf(stderr, "[agt] refine_host: first pass done at %.3f ms, %d frames to redo\n", since(), n_redo);
    if (n_redo > 0) {
      // compact the initial poses of the redo frames into their own job arrays and scatter the results back
      agt_jobs R;
      const int64_t j2 = (int64_t)n_redo * n_hyp;
      uint8_t* dr2;
      if ((rc = agt_scratch(ctx, SLOT_REDO_JOBS, layout_jobs(&R, nullptr, j2), reinterpret_cast<void**>(&dr2)))) return rc;
      layout_jobs(&R, dr2, j2);
      for (int i = 0; i < n_redo; ++i)
        AGT_CUDA(ctx, cudaMemcpyAsync(R.init + (int64_t)i * n_hyp * 6, h_init + (int64_t)ids[i] * n_hyp * 6, sizeof(double) * 6 * n_hyp,
                                      cudaMemcpyHostToDevice, st));
      AGT_CUDA(ctx, cudaEventRecord(ctx->ev[3], st));
      AGT_CUDA(ctx, cudaStreamWaitEvent(cp, ctx->ev[3], 0));
      d.kind = PASS_REDO;
      d.chunk = chunk < n_redo ? chunk : n_redo;
      d.rects.clear();
      for (int f : ids) d.rects.push_back({0, 0, w, h, f});
      if ((rc = refine_pass(ctx, d, R, buf))) return rc;
      for (int i = 0; i < n_redo; ++i) {
        const int64_t from = (int64_t)i * n_hyp, to = (int64_t)ids[i] * n_hyp;
        AGT_CUDA(ctx, cudaMemcpyAsync(J.pose + 6 * to, R.pose + 6 * from, sizeof(double) * 6 * n_hyp, cudaMemcpyDeviceToDevice, st));
        AGT_CUDA(ctx, cudaMemcpyAsync(J.cost + to, R.cost + from, sizeof(float) * n_hyp, cudaMemcpyDeviceToDevice, st));
        AGT_CUDA(ctx, cudaMemcpyAsync(J.n_valid + to, R.n_valid + from, sizeof(int32_t) * n_hyp, cudaMemcpyDeviceToDevice, st));
        AGT_CUDA(ctx, cudaMemcpyAsync(J.evals + to, R.evals + from, sizeof(int32_t) * n_hyp, cudaMemcpyDeviceToDevice, st));
        AGT_CUDA(ctx, cudaMemcpyAsync(J.status + to, R.status + from, (size_t)n_hyp, cudaMemcpyDeviceToDevice, st));
      }
    }
  }
  if (n_hyp > 1 && h_best) {
    if ((rc = agt_select_best(ctx, J.pose, J.cost, J.n_valid, n_hyp, d_best, nullptr, batch))) return rc;
    AGT_CUDA(ctx, cudaMemcpyAsync(h_best, d_best, sizeof(int32_t) * batch, cudaMemcpyDeviceToHost, st));
  }
  AGT_CUDA(ctx, cudaMemcpyAsync(h_pose, J.pose, sizeof(double) * 6 * jobs, cudaMemcpyDeviceToHost, st));
  if (h_cost) AGT_CUDA(ctx, cudaMemcpyAsync(h_cost, J.cost, sizeof(float) * jobs, cudaMemcpyDeviceToHost, st));
  if (h_n_valid) AGT_CUDA(ctx, cudaMemcpyAsync(h_n_valid, J.n_valid, sizeof(int32_t) * jobs, cudaMemcpyDeviceToHost, st));
  if (h_evals) AGT_CUDA(ctx, cudaMemcpyAsync(h_evals, J.evals, sizeof(int32_t) * jobs, cudaMemcpyDeviceToHost, st));
  if (h_status) AGT_CUDA(ctx, cudaMemcpyAsync(h_status, J.status, jobs, cudaMemcpyDeviceToHost, st));
  AGT_CUDA(ctx, cudaStreamSynchronize(st));
  if (trace) fprintf(stderr, "[agt] refine_host: done at %.3f ms\n", since());
  return AGT_OK;
} catch (const std::bad_alloc&) {            // the host lists of a call (ctx is set: nothing allocates before its check)
  AGT_FAIL(ctx, AGT_ERR_INVALID, "agt_refine_host: out of host memory");
}

extern "C" int agt_pose_covariance_host(agt_ctx* ctx, const uint8_t* h_frames, int w, int h, int levels, int batch, const double* h_init,
                                        const double* h_pose, int n_hyp, double* h_cov, double* h_info, float* h_sigma2,
                                        int32_t* h_n_valid, uint8_t* h_ok) {
  if (!ctx) return AGT_ERR_INVALID;
  if (!h_frames || !h_init || !h_pose || !h_cov || !h_ok || w < 1 || h < 1 || levels < 1 || levels > AGT_MAX_LEVELS || batch < 0 ||
      n_hyp < 1)
    AGT_FAIL(ctx, AGT_ERR_INVALID, "agt_pose_covariance_host: bad arguments");
  if (batch == 0) return AGT_OK;
  AGT_CUDA(ctx, cudaSetDevice(ctx->device));
  // whole frames, one pyramid for the batch (SLOT_CHUNK0), then the poses and the outputs (SLOT_JOBS)
  agt_pyramid p;
  const int64_t pyr_bytes = layout_pyramid(&p, nullptr, w, h, levels, batch);
  const int64_t jobs = (int64_t)batch * n_hyp;
  const int64_t o_pose = align_up(sizeof(double) * 6 * jobs, 256), o_cov = o_pose + o_pose, o_info = o_cov + align_up(sizeof(double) * 36 * jobs, 256),
                o_s2 = o_info + align_up(sizeof(double) * 36 * jobs, 256), o_nv = o_s2 + align_up(sizeof(float) * jobs, 256),
                o_ok = o_nv + align_up(sizeof(int32_t) * jobs, 256), total = o_ok + align_up(jobs, 256);
  uint8_t *dp, *d;
  int rc;
  if ((rc = agt_scratch(ctx, SLOT_CHUNK0, (size_t)pyr_bytes, reinterpret_cast<void**>(&dp)))) return rc;
  if ((rc = agt_scratch(ctx, SLOT_JOBS, (size_t)total, reinterpret_cast<void**>(&d)))) return rc;
  layout_pyramid(&p, dp, w, h, levels, batch);
  cudaStream_t st = ctx->stream;
  // level 0 rows of consecutive frames are consecutive (frame_stride = pitch * h): one 2-D copy for the batch
  AGT_CUDA(ctx, cudaMemcpy2DAsync(p.data[0], (size_t)p.pitch[0], h_frames, (size_t)w, (size_t)w, (size_t)h * batch,
                                  cudaMemcpyHostToDevice, st));
  AGT_CUDA(ctx, cudaMemcpyAsync(d, h_init, sizeof(double) * 6 * jobs, cudaMemcpyHostToDevice, st));
  AGT_CUDA(ctx, cudaMemcpyAsync(d + o_pose, h_pose, sizeof(double) * 6 * jobs, cudaMemcpyHostToDevice, st));
  if ((rc = agt_build_pyramid(ctx, &p, batch))) return rc;
  if ((rc = agt_pose_covariance(ctx, &p, reinterpret_cast<const double*>(d), reinterpret_cast<const double*>(d + o_pose), n_hyp, nullptr,
                                reinterpret_cast<double*>(d + o_cov), reinterpret_cast<double*>(d + o_info),
                                reinterpret_cast<float*>(d + o_s2), reinterpret_cast<int32_t*>(d + o_nv), d + o_ok, batch)))
    return rc;
  AGT_CUDA(ctx, cudaMemcpyAsync(h_cov, d + o_cov, sizeof(double) * 36 * jobs, cudaMemcpyDeviceToHost, st));
  if (h_info) AGT_CUDA(ctx, cudaMemcpyAsync(h_info, d + o_info, sizeof(double) * 36 * jobs, cudaMemcpyDeviceToHost, st));
  if (h_sigma2) AGT_CUDA(ctx, cudaMemcpyAsync(h_sigma2, d + o_s2, sizeof(float) * jobs, cudaMemcpyDeviceToHost, st));
  if (h_n_valid) AGT_CUDA(ctx, cudaMemcpyAsync(h_n_valid, d + o_nv, sizeof(int32_t) * jobs, cudaMemcpyDeviceToHost, st));
  AGT_CUDA(ctx, cudaMemcpyAsync(h_ok, d + o_ok, (size_t)jobs, cudaMemcpyDeviceToHost, st));
  AGT_CUDA(ctx, cudaStreamSynchronize(st));
  return AGT_OK;
}
