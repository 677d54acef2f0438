// N3 (SURVEY.md 8f): tag identification and detection on the device.
//
// The reference detects tags with the un-vendored swatbotics apriltag library (detect_pose.py:86-95 tag36h11; :368-371 detect;
// :389-400 decision_margin filter, corner order of transform_helper.py:56-59).  The frozen semantics here are those of
// oracle/tag_oracle.py, pinned to OpenCV's ArUco module (same family, DICT_APRILTAG_36h11) in the tests.
//
// agt_decode_tags - warp per quad: the 8x8 cells (6x6 data + black border) are sampled through the quad's homography (3x3
// bilinear samples per cell, two cells per lane), the threshold lies half way between the darkest and the brightest cell, the
// border may hold two wrong cells, and the 36 data bits are matched against the family over the four rotations (each lane
// tries every 32nd code word, popcount of the xor); returns id, rotation, Hamming distance and the mean distance of the cells
// from the threshold - the analogue of apriltag's decision_margin, which the reference compares with 50.
#include <cooperative_groups.h>
#include <algorithm>

#include "agt_common.cuh"

// Iteration cap of the detector's corner refinement (stop rule: a step below 1e-3 px or this many iterations).  A corner of a
// tag converges in 3-6 iterations; what runs longer is the corner of a quadrilateral that is no tag, or a corner bouncing
// between two float32 positions - and the launch lasts as long as its slowest corner.  With 10 the ids and corners of the probe
// frames are unchanged (scripts/tag_detect_probe.py) and the pass takes 32 instead of 57 us; cv2.aruco's own refinement stops
// far earlier (cornerRefinementMinAccuracy 0.1 px).
constexpr int TAG_SUBPIX_ITERS = 10;

namespace {

constexpr int CELLS = 8;
constexpr int TG_WARPS = 4;

struct Homography { double a, b, c, d, e, f, g, h; };

// unit square (s right, t down, (0,0) = top-left) -> quad given as (bottom-left, top-left, top-right, bottom-right)
__device__ __forceinline__ Homography square_to_quad(const float* q) {
  const double x3 = q[0], y3 = q[1], x0 = q[2], y0 = q[3], x1 = q[4], y1 = q[5], x2 = q[6], y2 = q[7];
  const double dx1 = x1 - x2, dx2 = x3 - x2, sx = x0 - x1 + x2 - x3;
  const double dy1 = y1 - y2, dy2 = y3 - y2, sy = y0 - y1 + y2 - y3;
  const double den = dx1 * dy2 - dx2 * dy1;
  Homography H;
  H.g = (sx * dy2 - dx2 * sy) / den;
  H.h = (dx1 * sy - sx * dy1) / den;
  H.a = x1 - x0 + H.g * x1; H.b = x3 - x0 + H.h * x3; H.c = x0;
  H.d = y1 - y0 + H.g * y1; H.e = y3 - y0 + H.h * y3; H.f = y0;
  return H;
}

// where the detector wants the quads that decode to a tag: per frame a counter and max_tags slots (out_n == NULL: nowhere)
struct TagSink {
  int32_t* out_n; int32_t* out_id; float* out_corners; float* out_margin; uint8_t* out_ham; int max_tags;
};

__global__ void __launch_bounds__(TG_WARPS * 32)
decode_tags_kernel(const uint8_t* __restrict__ img, int w, int h, int64_t pitch, int64_t stride, const float* __restrict__ quads,
                   const uint8_t* __restrict__ valid, const unsigned long long* __restrict__ codes, int n_codes, int32_t* __restrict__ id_out,
                   uint8_t* __restrict__ rot_out, uint8_t* __restrict__ ham_out, float* __restrict__ margin_out, int n_quads, int64_t total,
                   int max_hamming, const TagSink sink) {
  const int lane = threadIdx.x & 31;
  const int64_t gid = (int64_t)blockIdx.x * TG_WARPS + (threadIdx.x >> 5);
  if (gid >= total) return;
  int id = -1, rot = 0, ham = 255;
  float margin = 0.f;
  const float* q = quads + gid * 8;
  bool fin = true;
  for (int k = 0; k < 8; ++k) fin = fin && isfinite(q[k]);
  if ((valid == nullptr || valid[gid] != 0) && fin) {
    const uint8_t* f = img + (gid / n_quads) * stride;
    const Homography H = square_to_quad(q);
    double m[2];
    bool inside = true;
#pragma unroll
    for (int half = 0; half < 2; ++half) {
      const int cell = lane + 32 * half, r = cell >> 3, c = cell & 7;
      double acc = 0.0;
      for (int dt = -1; dt <= 1; ++dt)
        for (int ds = -1; ds <= 1; ++ds) {
          const double s = ((double)c + 0.5 + 0.25 * ds) / CELLS, t = ((double)r + 0.5 + 0.25 * dt) / CELLS;
          const double iw = 1.0 / (H.g * s + H.h * t + 1.0);
          const double x = (H.a * s + H.b * t + H.c) * iw, y = (H.d * s + H.e * t + H.f) * iw;
          const double fx0 = floor(x), fy0 = floor(y);
          if (!(fx0 >= 0.0 && fy0 >= 0.0 && fx0 + 1.0 < (double)w && fy0 + 1.0 < (double)h)) { inside = false; continue; }
          const int x0 = (int)fx0, y0 = (int)fy0;
          const double ax = x - fx0, ay = y - fy0;
          const uint8_t* p = f + (int64_t)y0 * pitch + x0;
          acc += (1.0 - ax) * (1.0 - ay) * (double)__ldg(p) + ax * (1.0 - ay) * (double)__ldg(p + 1) +
                 (1.0 - ax) * ay * (double)__ldg(p + pitch) + ax * ay * (double)__ldg(p + pitch + 1);
        }
      m[half] = acc / 9.0;
    }
    inside = __all_sync(0xffffffffu, inside);
    if (inside) {
      double lo = fmin(m[0], m[1]), hi = fmax(m[0], m[1]);
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) { lo = fmin(lo, __shfl_xor_sync(0xffffffffu, lo, o)); hi = fmax(hi, __shfl_xor_sync(0xffffffffu, hi, o)); }
      const double thr = 0.5 * (lo + hi);
      const unsigned b0 = __ballot_sync(0xffffffffu, m[0] > thr), b1 = __ballot_sync(0xffffffffu, m[1] > thr);
      const unsigned long long bits = (unsigned long long)b0 | ((unsigned long long)b1 << 32);      // bit r*8+c
      margin = (float)(agt_warp_sum(fabs(m[0] - thr) + fabs(m[1] - thr)) / 64.0);
      const unsigned long long border = 0xFF818181818181FFull;
      if (__popcll(bits & border) <= 2) {
        // data word of each rotation: grid[i][j] = data[src(i, j)], row-major, first cell = most significant bit
        unsigned long long word[4] = {0, 0, 0, 0};
#pragma unroll
        for (int rt = 0; rt < 4; ++rt)
          for (int i = 0; i < 6; ++i)
            for (int j = 0; j < 6; ++j) {
              const int sr = rt == 0 ? i : (rt == 1 ? 5 - j : (rt == 2 ? 5 - i : j));
              const int sc = rt == 0 ? j : (rt == 1 ? i : (rt == 2 ? 5 - j : 5 - i));
              word[rt] = (word[rt] << 1) | ((bits >> ((sr + 1) * 8 + sc + 1)) & 1ull);
            }
        unsigned best = 0xffffffffu;                    // hamming << 24 | rotation << 16 | id: the oracle's tie-breaking order
        for (int i = lane; i < n_codes; i += 32) {
          const unsigned long long code = codes[i];
#pragma unroll
          for (int rt = 0; rt < 4; ++rt) {
            const unsigned key = ((unsigned)__popcll(word[rt] ^ code) << 24) | ((unsigned)rt << 16) | (unsigned)i;
            best = min(best, key);
          }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) best = min(best, __shfl_xor_sync(0xffffffffu, best, o));
        ham = (int)(best >> 24);
        if (best != 0xffffffffu && ham <= max_hamming) { id = (int)(best & 0xffffu); rot = (int)((best >> 16) & 0xffu); }
      }
    }
  }
  if (lane == 0) {
    id_out[gid] = id;
    if (rot_out) rot_out[gid] = (uint8_t)rot;
    if (ham_out) ham_out[gid] = (uint8_t)(ham > 255 ? 255 : ham);
    if (margin_out) margin_out[gid] = margin;
  }
  if (sink.out_n != nullptr && id >= 0) {
    // the detector's list of tags, corners in the reference's order: the quad's corner k is the tag's corner (k + rot) mod 4
    const int64_t f = gid / n_quads;
    int slot = lane == 0 ? atomicAdd(&sink.out_n[f], 1) : 0;
    slot = __shfl_sync(0xffffffffu, slot, 0);
    if (slot < sink.max_tags) {
      const int64_t o = f * sink.max_tags + slot;
      if (lane < 8) sink.out_corners[o * 8 + lane] = q[2 * (((lane >> 1) - rot + 4) & 3) + (lane & 1)];
      if (lane == 0) {
        sink.out_id[o] = id;
        if (sink.out_margin) sink.out_margin[o] = margin;
        if (sink.out_ham) sink.out_ham[o] = (uint8_t)ham;
      }
    }
  }
}

}  // namespace

extern "C" int agt_set_tag_family(agt_ctx* ctx, const uint64_t* h_codes, int n_codes) {
  if (!ctx) return AGT_ERR_INVALID;
  if (!h_codes || n_codes < 1 || n_codes > 65535) AGT_FAIL(ctx, AGT_ERR_INVALID, "agt_set_tag_family: 1..65535 code words of 36 bits");
  AGT_CUDA(ctx, cudaSetDevice(ctx->device));
  if (ctx->d_tag_codes) { AGT_CUDA(ctx, cudaStreamSynchronize(ctx->stream)); cudaFree(ctx->d_tag_codes); ctx->d_tag_codes = nullptr; }
  AGT_CUDA(ctx, cudaMalloc(reinterpret_cast<void**>(&ctx->d_tag_codes), sizeof(uint64_t) * (size_t)n_codes));
  AGT_CUDA(ctx, cudaMemcpy(ctx->d_tag_codes, h_codes, sizeof(uint64_t) * (size_t)n_codes, cudaMemcpyHostToDevice));
  ctx->n_tag_codes = n_codes;
  return AGT_OK;
}

extern "C" int agt_set_tag_threshold(agt_ctx* ctx, int mode) {
  if (!ctx) return AGT_ERR_INVALID;
  if (mode < 0 || mode > 2) AGT_FAIL(ctx, AGT_ERR_INVALID, "agt_set_tag_threshold: mode 0 (auto), 1 (per window) or 2 (local white level)");
  ctx->tag_threshold = mode;
  return AGT_OK;
}

static int decode_tags(agt_ctx* ctx, const uint8_t* d_gray, int w, int h, int64_t pitch, int64_t stride, const float* d_quads,
                       const uint8_t* d_valid, int32_t* d_id, uint8_t* d_rotation, uint8_t* d_hamming, float* d_margin, int batch,
                       int n_quads, int max_hamming, const TagSink& sink) {
  if (!ctx) return AGT_ERR_INVALID;
  if ((int64_t)batch * n_quads == 0) return AGT_OK;
  if (!ctx->d_tag_codes) AGT_FAIL(ctx, AGT_ERR_NOT_READY, "agt_decode_tags: call agt_set_tag_family first");
  if (!d_gray || !d_quads || !d_id || batch < 0 || n_quads < 0 || w < 2 || h < 2 || pitch < w || max_hamming < 0 || max_hamming > 10)
    AGT_FAIL(ctx, AGT_ERR_INVALID, "agt_decode_tags: bad arguments");
  const int64_t total = (int64_t)batch * n_quads, blocks = (total + TG_WARPS - 1) / TG_WARPS;
  if (blocks > 0x7fffffffLL) AGT_FAIL(ctx, AGT_ERR_INVALID, "agt_decode_tags: batch too large");
  decode_tags_kernel<<<(unsigned)blocks, TG_WARPS * 32, 0, ctx->stream>>>(d_gray, w, h, pitch, stride, d_quads, d_valid,
                                                                          reinterpret_cast<const unsigned long long*>(ctx->d_tag_codes),
                                                                          ctx->n_tag_codes, d_id, d_rotation, d_hamming, d_margin, n_quads, total,
                                                                          max_hamming, sink);
  AGT_LAUNCH_CHECK(ctx);
  return AGT_OK;
}

extern "C" int agt_decode_tags(agt_ctx* ctx, const uint8_t* d_gray, int w, int h, int64_t pitch, int64_t stride, const float* d_quads,
                               const uint8_t* d_valid, int32_t* d_id, uint8_t* d_rotation, uint8_t* d_hamming, float* d_margin, int batch,
                               int n_quads, int max_hamming) {
  return decode_tags(ctx, d_gray, w, h, pitch, stride, d_quads, d_valid, d_id, d_rotation, d_hamming, d_margin, batch, n_quads, max_hamming,
                     TagSink{nullptr, nullptr, nullptr, nullptr, nullptr, 0});
}

// =====================================================================================================================
// agt_detect_tags: quads of dark square regions -> corner refinement -> identification, for a batch of gray frames.
//
//   threshold   dark <=> gray < lo + 0.35 (hi - lo).  lo = the darkest pixel of the search window.  hi = the brightest pixel of
//               the window (one threshold per window: a tracking window is a few hundred pixels wide, which is local already),
//               or - whole frames, agt_set_tag_threshold - the brightest pixel of the 3 x 3 tiles of 32 x 32 pixels around the
//               pixel: the local white level.  Uneven lighting is a smooth gain on the scene: it moves white by its full
//               factor and black by next to nothing, so the threshold follows white and keeps the window's black.  (Taking
//               lo from the neighbourhood as well - the adaptive threshold of the CPU detectors - turns mid-gray background
//               next to a white quiet zone into dark frames around every tag that the later passes would have to discard.)
//   components  4-connected components of the dark pixels: a mask word per 32-pixel item and a list of the non-empty items,
//               union-find over the runs of a frame in shared memory (ccl_runs_kernel; cluttered frames: union-find over
//               the pixels in global memory)
//   quad        per component: area, centroid; the boundary pixel farthest from the centroid (c0), the one farthest from
//               c0 (c2), and the ones farthest from the line c0 c2 on either side (c1, c3) - the four corners of a convex
//               quadrilateral whatever its orientation; components that are too small, touch the frame or are not
//               quadrilateral (area far from the quad's) are dropped
//   refine      agt_corner_subpix (cv::cornerSubPix) on the four corners, then agt_decode_tags; quads that decode to a tag
//               are written in the reference's corner order (rolled by the decoded rotation)
// =====================================================================================================================
namespace {

constexpr int MAX_COMPONENTS = 4096;      // per frame, components of area >= 48 (no smaller one can become a quad); what does not fit is ignored (counted)

struct CompStats {
  int area;
  int x0, y0, x1, y1;
  unsigned long long sx, sy;
  unsigned long long far0, far2, side_p, side_n;      // (ordered float key << 32) | pixel index
};

__device__ __forceinline__ unsigned long long far_key(float v, int idx) {
  return ((unsigned long long)__float_as_uint(fmaxf(v, 0.f)) << 32) | (unsigned)idx;       // non-negative floats order like integers
}

// search window of a frame: the whole frame, or the part of it inside the frame's rectangle (x0, y0, x1, y1; an empty rectangle
// means the whole frame; the left edge is moved to a multiple of 16 pixels so that rows can be read as aligned words).  Pixel
// index i of a window runs row by row over the window; labels are indexed the same way.
struct Win { int x0, y0, ww, hh; };
__device__ __forceinline__ Win frame_window(const int32_t* rects, int rect_stride, int f, int w, int h) {
  Win q = {0, 0, w, h};
  if (rects != nullptr) {
    const int32_t* r = rects + (int64_t)f * rect_stride;
    const int x0 = max(r[0], 0) & ~15, y0 = max(r[1], 0), x1 = min(r[2], w), y1 = min(r[3], h);
    if (x1 > x0 && y1 > y0) { q.x0 = x0; q.y0 = y0; q.ww = x1 - x0; q.hh = y1 - y0; }
  }
  return q;
}
#define AGT_WIN_ARGS const int32_t* __restrict__ rects, int rect_stride

// Layout of the component passes.  A window row is cut into 32-pixel items (item = row * chunks + chunk); ccl_init_kernel
// writes one mask word per item (bit b = pixel 32 chunk + b is dark) and appends the non-empty items (a few percent of a frame,
// 10-15 % of a search window) to a list.  Every later pass runs a warp per list entry, lane = pixel: which neighbours are dark
// is bit arithmetic on the mask words of the neighbouring items, labels are read and written at dark pixels only.
#define AGT_WARP_SETUP                                                                                                 \
  const int f = blockIdx.y;                                                                                            \
  const Win win = frame_window(rects, rect_stride, f, w, h);                                                           \
  const int lane = threadIdx.x & 31, chunks = (win.ww + 31) >> 5;                                                      \
  const int warp0 = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), nwarps = gridDim.x * (blockDim.x >> 5);
struct Entry { int item, y, ch, x, i; unsigned m; bool dark; };
__device__ __forceinline__ Entry load_entry(const int2* __restrict__ E, int e, int n, int chunks, int ww, int lane) {
  Entry t;
  const int2 v = e < n ? E[e] : make_int2(0, 0);
  t.item = v.x; t.m = (unsigned)v.y;
  t.y = t.item / chunks; t.ch = t.item - t.y * chunks; t.x = t.ch * 32 + lane; t.i = t.y * ww + t.x;
  t.dark = (t.m >> lane) & 1u;
  return t;
}

// rows of the window can be read as 16-byte words (the window's left edge is a multiple of 16 pixels by construction)
__device__ __forceinline__ bool rows_aligned16(const uint8_t* p, int64_t pitch, const Win& win) {
  return (reinterpret_cast<uintptr_t>(p) & 15) == 0 && (pitch & 15) == 0 && (win.x0 & 15) == 0;
}

// four pixels of a row as one word (x counts from the left edge of the window; pixels beyond the window read as 0)
__device__ __forceinline__ uint32_t load_px4(const uint8_t* __restrict__ row, int x, int ww, bool aligned) {
  if (aligned) return *reinterpret_cast<const uint32_t*>(row + x);
  uint32_t v = 0;
#pragma unroll
  for (int k = 0; k < 4; ++k) if (x + k < ww) v |= (uint32_t)row[x + k] << (8 * k);
  return v;
}

__global__ void frame_minmax_kernel(const uint8_t* __restrict__ img, int w, int h, int64_t pitch, int64_t stride, AGT_WIN_ARGS,
                                    int* __restrict__ lohi) {
  const uint8_t* p = img + blockIdx.y * stride;
  const bool aligned = (reinterpret_cast<uintptr_t>(p) & 3) == 0 && (pitch & 3) == 0;
  AGT_WARP_SETUP
  (void)chunks;
  const int gchunks = (win.ww + 127) >> 7, gitems = gchunks * win.hh;
  uint32_t lo4 = 0xffffffffu, hi4 = 0u;
  if (aligned && (reinterpret_cast<uintptr_t>(p) & 15) == 0 && (pitch & 15) == 0 && (win.x0 & 15) == 0) {
    // sixteen pixels per lane: a warp reads 512 pixels of a row per load
    const int wch = (win.ww + 511) >> 9, witems = wch * win.hh;
    for (int base = warp0 * 2; base < witems; base += nwarps * 2) {
#pragma unroll
      for (int k = 0; k < 2; ++k) {
        const int g = base + k, y = g / wch, x = (g - y * wch) * 512 + 16 * lane;
        if (g < witems && x < win.ww) {
          const uint4 v = *reinterpret_cast<const uint4*>(p + (int64_t)(win.y0 + y) * pitch + win.x0 + x);
          const uint32_t q[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const int nv = min(4, win.ww - x - 4 * j);
            if (nv <= 0) continue;
            const uint32_t inv = nv < 4 ? 0xffffffffu << (8 * nv) : 0u;
            lo4 = __vminu4(lo4, q[j] | inv); hi4 = __vmaxu4(hi4, q[j] & ~inv);
          }
        }
      }
    }
  } else {
    for (int base = warp0 * 4; base < gitems; base += nwarps * 4) {
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int g = base + k, y = g / gchunks, x = (g - y * gchunks) * 128 + 4 * lane;
        if (g < gitems && x < win.ww) {
          const uint32_t v = load_px4(p + (int64_t)(win.y0 + y) * pitch + win.x0, x, win.ww, aligned);
          const int nv = min(4, win.ww - x);
          const uint32_t inv = nv < 4 ? 0xffffffffu << (8 * nv) : 0u;
          lo4 = __vminu4(lo4, v | inv); hi4 = __vmaxu4(hi4, v & ~inv);
        }
      }
    }
  }
  int lo = min(min(lo4 & 0xff, (lo4 >> 8) & 0xff), min((lo4 >> 16) & 0xff, lo4 >> 24));
  int hi = max(max(hi4 & 0xff, (hi4 >> 8) & 0xff), max((hi4 >> 16) & 0xff, hi4 >> 24));
  lo = __reduce_min_sync(0xffffffffu, lo); hi = __reduce_max_sync(0xffffffffu, hi);
  if ((threadIdx.x & 31) == 0 && lo <= hi) { atomicMax(&lohi[2 * blockIdx.y], 255 - lo); atomicMax(&lohi[2 * blockIdx.y + 1], hi); }
}

__device__ __forceinline__ int threshold_of(int lo, int hi) {
  return hi - lo < 40 ? -1 : lo + (35 * (hi - lo)) / 100;              // no contrast, no dark pixels
}
// lohi[2 f] = 255 - the darkest pixel, lohi[2 f + 1] = the brightest: both grow from zeroed memory by atomicMax
__device__ __forceinline__ int frame_lo(const int* lohi, int f) { return 255 - lohi[2 * f]; }
__device__ __forceinline__ int frame_threshold(const int* lohi, int f) { return threshold_of(frame_lo(lohi, f), lohi[2 * f + 1]); }

// Local white level: the brightest pixel of every 32 x 32 tile of a window (tile (ty, tx) = rows 32 ty.., item tx of the row), and
// the window's darkest / brightest pixel as frame_minmax_kernel leaves them.  A warp takes four tiles of a tile row: 128 pixels
// of a row per load, the eight lanes of a tile put their maxima together.
constexpr int TILE = 32;
__global__ void tile_max_kernel(const uint8_t* __restrict__ img, int w, int h, int64_t pitch, int64_t stride, AGT_WIN_ARGS,
                                int* __restrict__ lohi, uint8_t* __restrict__ tile_hi, int64_t tile_stride) {
  const uint8_t* p = img + blockIdx.y * stride;
  const bool aligned = (reinterpret_cast<uintptr_t>(p) & 3) == 0 && (pitch & 3) == 0;
  AGT_WARP_SETUP
  uint8_t* T = tile_hi + f * tile_stride;
  const int gchunks = (win.ww + 127) >> 7, trows = (win.hh + TILE - 1) / TILE;
  uint32_t wlo4 = 0xffffffffu, whi4 = 0u;
  if (rows_aligned16(p, pitch, win)) {
    // sixteen pixels per lane: a warp takes 512 pixels of a tile row, two lanes make a tile
    const int wch = (win.ww + 511) >> 9;
    for (int g = warp0; g < wch * trows; g += nwarps) {
      const int ty = g / wch, c = g - ty * wch, x = c * 512 + 16 * lane;
      uint32_t lo4 = 0xffffffffu, hi4 = 0u;
      if (x < win.ww) {
        uint32_t inv[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) { const int nv = min(4, max(win.ww - x - 4 * j, 0)); inv[j] = nv < 4 ? 0xffffffffu << (8 * nv) : 0u; }
        const uint8_t* row = p + (int64_t)(win.y0 + ty * TILE) * pitch + win.x0 + x;
        const int ny = min(win.hh, (ty + 1) * TILE) - ty * TILE;
#pragma unroll 4
        for (int y = 0; y < ny; ++y) {
          const uint4 v = *reinterpret_cast<const uint4*>(row + (int64_t)y * pitch);
          lo4 = __vminu4(lo4, __vminu4(__vminu4(v.x | inv[0], v.y | inv[1]), __vminu4(v.z | inv[2], v.w | inv[3])));
          hi4 = __vmaxu4(hi4, __vmaxu4(__vmaxu4(v.x & ~inv[0], v.y & ~inv[1]), __vmaxu4(v.z & ~inv[2], v.w & ~inv[3])));
        }
      }
      wlo4 = __vminu4(wlo4, lo4); whi4 = __vmaxu4(whi4, hi4);
      hi4 = __vmaxu4(hi4, __shfl_xor_sync(0xffffffffu, hi4, 1));
      const int tx = c * 16 + (lane >> 1);
      if ((lane & 1) == 0 && tx < chunks) T[ty * chunks + tx] = (uint8_t)max(max(hi4 & 0xff, (hi4 >> 8) & 0xff), max((hi4 >> 16) & 0xff, hi4 >> 24));
    }
  } else
  for (int g = warp0; g < gchunks * trows; g += nwarps) {
    const int ty = g / gchunks, gc = g - ty * gchunks, x = gc * 128 + 4 * lane;
    uint32_t lo4 = 0xffffffffu, hi4 = 0u;
    if (x < win.ww) {
      const int nv = min(4, win.ww - x);
      const uint32_t inv = nv < 4 ? 0xffffffffu << (8 * nv) : 0u;
      const int y1 = min(win.hh, (ty + 1) * TILE);
#pragma unroll 8
      for (int y = ty * TILE; y < y1; ++y) {
        const uint32_t v = load_px4(p + (int64_t)(win.y0 + y) * pitch + win.x0, x, win.ww, aligned);
        lo4 = __vminu4(lo4, v | inv); hi4 = __vmaxu4(hi4, v & ~inv);
      }
    }
    wlo4 = __vminu4(wlo4, lo4); whi4 = __vmaxu4(whi4, hi4);
    hi4 = __vmaxu4(hi4, __shfl_xor_sync(0xffffffffu, hi4, 1)); hi4 = __vmaxu4(hi4, __shfl_xor_sync(0xffffffffu, hi4, 2));
    hi4 = __vmaxu4(hi4, __shfl_xor_sync(0xffffffffu, hi4, 4));
    const int tx = gc * 4 + (lane >> 3);
    if ((lane & 7) == 0 && tx < chunks) T[ty * chunks + tx] = (uint8_t)max(max(hi4 & 0xff, (hi4 >> 8) & 0xff), max((hi4 >> 16) & 0xff, hi4 >> 24));
  }
  int lo = min(min(wlo4 & 0xff, (wlo4 >> 8) & 0xff), min((wlo4 >> 16) & 0xff, wlo4 >> 24));
  int hi = max(max(whi4 & 0xff, (whi4 >> 8) & 0xff), max((whi4 >> 16) & 0xff, whi4 >> 24));
  lo = __reduce_min_sync(0xffffffffu, lo); hi = __reduce_max_sync(0xffffffffu, hi);
  if (lane == 0 && lo <= hi) { atomicMax(&lohi[2 * f], 255 - lo); atomicMax(&lohi[2 * f + 1], hi); }
}

// Threshold, mask words, list of non-empty items.  A warp reads 128 pixels of a row (four per lane); the eight lanes of an item put
// their dark bits together (rows readable as 16-byte words: sixteen pixels per lane, two lanes per item).  No pixel labels are
// written here: the common path works on runs (ccl_runs_kernel), and a frame that overflows its tables gets its labels there.
__global__ void ccl_init_kernel(const uint8_t* __restrict__ img, int w, int h, int64_t pitch, int64_t stride, AGT_WIN_ARGS,
                                const int* __restrict__ lohi, const uint8_t* __restrict__ tile_hi, int64_t tile_stride,
                                uint32_t* __restrict__ mask, int64_t mask_stride,
                                int* __restrict__ n_entries, int2* __restrict__ entries, int* __restrict__ entry_of) {
  const uint8_t* p = img + blockIdx.y * stride;
  const bool aligned = (reinterpret_cast<uintptr_t>(p) & 3) == 0 && (pitch & 3) == 0;
  const int frame_thr = frame_threshold(lohi, blockIdx.y), black = frame_lo(lohi, blockIdx.y);
  const uint8_t* T = tile_hi ? tile_hi + blockIdx.y * tile_stride : nullptr;
  uint32_t* M = mask + blockIdx.y * mask_stride;
  int2* E = entries + blockIdx.y * mask_stride;
  int* P = entry_of + blockIdx.y * mask_stride;        // position of a non-empty item in the list
  AGT_WARP_SETUP
  if (rows_aligned16(p, pitch, win)) {
    // Sixteen pixels per lane, two lanes per item; a warp takes 512 pixels of INIT_ROWS (1-16) consecutive rows: the threshold of an item
    // (nine tile maxima with the local white level) is formed once for those rows, the rows' loads do not depend on each other.
    // Dark bits of four pixels: per-byte compare, then the bytes' top bits gathered by one multiplication.
    const int wch = (win.ww + 511) >> 9, half = lane & 1;
    int INIT_ROWS = 16;                                  // a divisor of TILE; fewer rows per warp where that leaves warps without work
    while (INIT_ROWS > 1 && wch * ((win.hh + INIT_ROWS - 1) / INIT_ROWS) < nwarps) INIT_ROWS >>= 1;
    const int rgroups = (win.hh + INIT_ROWS - 1) / INIT_ROWS;
    for (int g = warp0; g < wch * rgroups; g += nwarps) {
      const int rg = g / wch, c = g - rg * wch, x = c * 512 + 16 * lane, ch = c * 16 + (lane >> 1);
      int thr = frame_thr;
      if (T != nullptr) {
        const int trows = (win.hh + TILE - 1) / TILE, ty = rg * INIT_ROWS / TILE, tx = min(ch, chunks - 1);
        int hi = 0;
#pragma unroll
        for (int k = 0; k < 5; ++k) {                                              // neighbours 0, 2, 4, 6, 8 / 1, 3, 5, 7 of the 3 x 3
          const int nb = min(2 * k + half, 8), dy = nb / 3 - 1, dx = nb - (nb / 3) * 3 - 1;
          hi = max(hi, (int)T[min(max(ty + dy, 0), trows - 1) * chunks + min(max(tx + dx, 0), chunks - 1)]);
        }
        hi = max(hi, __shfl_xor_sync(0xffffffffu, hi, 1));
        thr = threshold_of(black, hi);
      }
      const uint32_t thr4 = (uint32_t)max(thr, 0) * 0x01010101u;
      const int nv = min(16, win.ww - x);
      const uint32_t keep = nv >= 16 ? 0xffffu : (nv <= 0 ? 0u : (1u << nv) - 1u);
      const uint8_t* row = p + (int64_t)(win.y0 + rg * INIT_ROWS) * pitch + win.x0 + x;
      const int ny = min(win.hh, (rg + 1) * INIT_ROWS) - rg * INIT_ROWS;
#pragma unroll 4
      for (int yo = 0; yo < ny; ++yo) {
        uint4 v = make_uint4(~0u, ~0u, ~0u, ~0u);
        if (nv > 0) v = *reinterpret_cast<const uint4*>(row + (int64_t)yo * pitch);
        const uint32_t w4[4] = {v.x, v.y, v.z, v.w};
        unsigned m16 = 0;
#pragma unroll
        for (int j = 0; j < 4; ++j) m16 |= (((__vcmpltu4(w4[j], thr4) & 0x80808080u) * 0x00204081u) >> 28) << (4 * j);
        m16 &= keep;
        const unsigned other = __shfl_xor_sync(0xffffffffu, m16, 1);
        const unsigned m = half ? (other | (m16 << 16)) : (m16 | (other << 16));
        const int y = rg * INIT_ROWS + yo, item = y * chunks + ch;
        if (!half && ch < chunks) {
          M[item] = m;
          if (m != 0) {
            const int pos = atomicAdd(&n_entries[f], 1);
            E[pos] = make_int2(item, (int)m);
            P[item] = pos;
          }
        }
      }
    }
    return;
  }
  const int gchunks = (win.ww + 127) >> 7, gitems = gchunks * win.hh;
  const int sub = lane & 7, q = lane >> 3;
  for (int base = warp0 * 2; base < gitems; base += nwarps * 2) {
    uint32_t v[2];
    int yy[2], gc[2];
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      const int g = base + k;
      yy[k] = g / gchunks; gc[k] = g - yy[k] * gchunks;
      const int x = gc[k] * 128 + 4 * lane;
      v[k] = g < gitems && x < win.ww ? load_px4(p + (int64_t)(win.y0 + yy[k]) * pitch + win.x0, x, win.ww, aligned) : 0xffffffffu;
    }
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      const int x = gc[k] * 128 + 4 * lane;
      int thr = frame_thr;
      if (T != nullptr) {
        // local white level: the brightest of the 3 x 3 tiles around the item's tile, one neighbour per lane of the item
        const int trows = (win.hh + TILE - 1) / TILE, ty = min(yy[k], win.hh - 1) / TILE, tx = min(gc[k] * 4 + q, chunks - 1);
        const int dy = sub / 3 - 1, dx = sub - (sub / 3) * 3 - 1;                  // sub 0..7: eight neighbours; sub 0 adds (+1, +1)
        int hi = T[min(max(ty + dy, 0), trows - 1) * chunks + min(max(tx + dx, 0), chunks - 1)];
        if (sub == 0) hi = max(hi, (int)T[min(ty + 1, trows - 1) * chunks + min(tx + 1, chunks - 1)]);
        hi = max(hi, __shfl_xor_sync(0xffffffffu, hi, 1)); hi = max(hi, __shfl_xor_sync(0xffffffffu, hi, 2));
        hi = max(hi, __shfl_xor_sync(0xffffffffu, hi, 4));
        thr = threshold_of(black, hi);
      }
      unsigned nib = 0;
#pragma unroll
      for (int b = 0; b < 4; ++b) nib |= (x + b < win.ww && (int)((v[k] >> (8 * b)) & 0xffu) < thr) ? 1u << b : 0u;
      if (base + k >= gitems) nib = 0;
      unsigned m = nib << (4 * sub);
      m |= __shfl_xor_sync(0xffffffffu, m, 1); m |= __shfl_xor_sync(0xffffffffu, m, 2); m |= __shfl_xor_sync(0xffffffffu, m, 4);
      const int ch = gc[k] * 4 + q;
      if (base + k >= gitems || ch >= chunks) continue;
      const int item = yy[k] * chunks + ch;
      if (sub == 0) {
        M[item] = m;
        if (m != 0) {
          const int pos = atomicAdd(&n_entries[f], 1);
          E[pos] = make_int2(item, (int)m);
          P[item] = pos;
        }
      }
    }
  }
}

// a root is a pixel that points at itself, or - once ccl_flatten_number_kernel has been there - holds a negative component code
__device__ __forceinline__ int ccl_find(const int* L, int i) {
  int r = i;
  while (true) { const int p = L[r]; if (p == r || p < 0) return r; r = p; }
}
__device__ __forceinline__ void ccl_union(int* L, int a, int b) {
  while (true) {
    a = ccl_find(L, a); b = ccl_find(L, b);
    if (a == b) return;
    if (a < b) { const int t = a; a = b; b = t; }          // link the larger root below the smaller one
    const int old = atomicMin(&L[a], b);
    if (old == a) return;
    a = old;
  }
}

// Components of a frame in one CTA, in shared memory.  The unit is a run: a maximal row of dark pixels inside one item (a few
// hundred to a few thousand per search window).  Runs are numbered by a prefix sum over the list entries, joined - with the run
// left of them in the neighbouring item, with the runs above them - by union-find on a table in shared memory (the chains a tall
// component builds are walked at shared-memory latency: the same walk through global memory was three quarters of the
// detector's component time) and roots get their component number.  What leaves the kernel is the component code of every run:
// no pixel label is written or read on this path.  A frame with more entries or runs than the tables hold is flagged and goes
// through ccl_merge_kernel, ccl_area_kernel and ccl_flatten_number_kernel instead (which return at once for every other frame)
// and carries its codes in the pixel labels.
constexpr int RUNS_THREADS = 1024, RUNS_ENT_PER = 4, RUNS_ENT_CAP = RUNS_ENT_PER * RUNS_THREADS, RUNS_RUN_CAP = 6 * RUNS_THREADS;

// find with path halving: every node on the way is pointed at its grandparent.  Safe next to concurrent unions - a node that is
// not a root never becomes one again and is written by nobody but such walks, and any ancestor is a valid parent.
__device__ __forceinline__ int run_find(int* parent, int i) {
  int r = i, p = parent[r];
  while (p != r) {
    const int g = parent[p];
    if (g != p) parent[r] = g;
    r = p; p = g;
  }
  return r;
}
__device__ __forceinline__ void run_union(int* parent, int a, int b) {
  while (true) {
    a = run_find(parent, a); b = run_find(parent, b);
    if (a == b) return;
    if (a < b) { const int t = a; a = b; b = t; }
    const int old = atomicMin(&parent[a], b);
    if (old == a) return;
    a = old;
  }
}
// index, inside its item, of the run that holds bit b (starts = the first bits of the item's runs)
__device__ __forceinline__ int run_index(unsigned starts, int b) { return __popc(starts & ((2u << b) - 1u)) - 1; }

__global__ void __launch_bounds__(RUNS_THREADS, 1)
ccl_runs_kernel(int w, int h, AGT_WIN_ARGS, const uint32_t* __restrict__ mask, int64_t mask_stride,
                const int* __restrict__ n_entries, const int2* __restrict__ entries, const int* __restrict__ entry_of, int* __restrict__ n_comp,
                CompStats* __restrict__ stats, uint8_t* __restrict__ overflow, int* __restrict__ run_code, int* __restrict__ ent_base,
                int* __restrict__ label, int2* __restrict__ area_scratch) {
  __shared__ int s_parent[RUNS_RUN_CAP];
  __shared__ int s_base[RUNS_ENT_CAP];
  __shared__ int s_warp[RUNS_THREADS / 32];
  __shared__ int s_total;
  const int f = blockIdx.x, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const Win win = frame_window(rects, rect_stride, f, w, h);
  const int chunks = (win.ww + 31) >> 5;
  const uint32_t* M = mask + f * mask_stride;
  const int2* E = entries + f * mask_stride;
  const int* P = entry_of + f * mask_stride;
  const int n = n_entries[f];
  // A frame that does not fit the tables goes through the pixel-level union-find (ccl_merge_kernel ...), which wants every dark
  // pixel labelled with the first pixel of its run inside the item - a run is then one tree of depth 1 and the merge pass joins
  // runs, not pixels.  Only such frames pay for those labels.  The area counter of each run's first pixel (ccl_area_kernel) starts
  // at zero here.
  auto overflow_exit = [&]() {
    int* L = label + (int64_t)f * w * h;
    int* A = reinterpret_cast<int*>(area_scratch + (int64_t)f * w * h);
    for (int e = tid; e < n; e += RUNS_THREADS) {
      const int2 v = E[e];
      const int y = v.x / chunks, i0 = y * win.ww + (v.x - y * chunks) * 32;
      const unsigned m = (unsigned)v.y;
      unsigned mm = m;
      while (mm) {
        const int bit = __ffs(mm) - 1;
        mm &= mm - 1;
        const unsigned zeros_below = ~m & ((1u << bit) - 1u);
        L[i0 + bit] = i0 + (zeros_below ? 32 - __clz(zeros_below) : 0);
        if (bit == 0 || !((m >> (bit - 1)) & 1u)) A[i0 + bit] = 0;
      }
    }
    if (tid == 0) overflow[f] = 1;
  };
  if (n > RUNS_ENT_CAP) { overflow_exit(); return; }
  // ---- runs per entry, exclusive prefix sum (RUNS_ENT_PER consecutive entries per thread)
  int cnt[RUNS_ENT_PER], sum = 0;
#pragma unroll
  for (int k = 0; k < RUNS_ENT_PER; ++k) {
    const int e = tid * RUNS_ENT_PER + k;
    const unsigned m = e < n ? (unsigned)E[e].y : 0u;
    cnt[k] = __popc(m & ~(m << 1));
    sum += cnt[k];
  }
  int incl = sum;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) { const int v = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += v; }
  if (lane == 31) s_warp[wid] = incl;
  __syncthreads();
  if (wid == 0) {
    int v = lane < RUNS_THREADS / 32 ? s_warp[lane] : 0, iv = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int u = __shfl_up_sync(0xffffffffu, iv, o); if (lane >= o) iv += u; }
    if (lane < RUNS_THREADS / 32) s_warp[lane] = iv - v;
    if (lane == RUNS_THREADS / 32 - 1) s_total = iv;
  }
  __syncthreads();
  const int total = s_total;
  if (total > RUNS_RUN_CAP) { overflow_exit(); return; }
  {
    int run = s_warp[wid] + incl - sum;
#pragma unroll
    for (int k = 0; k < RUNS_ENT_PER; ++k) { s_base[tid * RUNS_ENT_PER + k] = run; run += cnt[k]; }
  }
  for (int r = tid; r < total; r += RUNS_THREADS) s_parent[r] = r;
  __syncthreads();
  // ---- joins, a thread per entry
  for (int e = tid; e < n; e += RUNS_THREADS) {
    const int2 v = E[e];
    const int item = v.x, y = item / chunks, ch = item - y * chunks;
    const unsigned m = (unsigned)v.y;
    const unsigned up = y > 0 ? M[item - chunks] : 0u, lw = ch > 0 ? M[item - 1] : 0u, ulw = ch > 0 && y > 0 ? M[item - chunks - 1] : 0u;
    const unsigned starts = m & ~(m << 1), base = (unsigned)s_base[e];
    if ((m & 1u) && (lw >> 31)) {
      const int pl = P[item - 1];
      run_union(s_parent, (int)base, s_base[pl] + __popc(lw & ~(lw << 1)) - 1);          // the last run of the item on the left
    }
    unsigned join = m & up & ~(((m << 1) | (lw >> 31)) & ((up << 1) | (ulw >> 31)));      // first column where a run meets a run above
    if (join) {
      const int ub = s_base[P[item - chunks]];
      const unsigned ustarts = up & ~(up << 1);
      while (join) {
        const int b = __ffs(join) - 1;
        join &= join - 1;
        run_union(s_parent, (int)base + run_index(starts, b), ub + run_index(ustarts, b));
      }
    }
  }
  __syncthreads();
  // ---- roots; every run points at its root, a root holds -1 - its area
  int root[RUNS_RUN_CAP / RUNS_THREADS];
#pragma unroll
  for (int k = 0; k < RUNS_RUN_CAP / RUNS_THREADS; ++k) {
    const int r = tid + k * RUNS_THREADS;
    root[k] = r < total ? run_find(s_parent, r) : -1;
  }
  __syncthreads();
#pragma unroll
  for (int k = 0; k < RUNS_RUN_CAP / RUNS_THREADS; ++k) {
    const int r = tid + k * RUNS_THREADS;
    if (r < total) s_parent[r] = root[k] == r ? -1 : root[k];
  }
  __syncthreads();
  for (int e = tid; e < n; e += RUNS_THREADS) {
    unsigned mm = (unsigned)E[e].y;
    int r = s_base[e];
    while (mm) {
      const int a = __ffs(mm) - 1;
      const unsigned t = mm >> a;
      const int len = t == 0xffffffffu ? 32 : __ffs(~t) - 1;
      mm &= len == 32 ? 0u : ~(((1u << len) - 1u) << a);
      const int p = s_parent[r];
      atomicSub(&s_parent[p < 0 ? r : p], len);
      ++r;
    }
  }
  __syncthreads();
  // ---- component numbers, codes: only a component that can become a quad (area >= 48, as far_pass and emit_quad ask) takes
  // one of the MAX_COMPONENTS numbers, so that specks do not crowd out the tags
#pragma unroll
  for (int k = 0; k < RUNS_RUN_CAP / RUNS_THREADS; ++k) {
    const int r = tid + k * RUNS_THREADS;
    if (r < total && root[k] == r) {
      const int c = -1 - s_parent[r] >= 48 ? atomicAdd(&n_comp[f], 1) : MAX_COMPONENTS;
      if (c < MAX_COMPONENTS) {
        CompStats& s = stats[(int64_t)f * MAX_COMPONENTS + c];
        s.area = 0; s.x0 = win.ww; s.y0 = win.hh; s.x1 = -1; s.y1 = -1; s.sx = 0; s.sy = 0; s.far0 = 0; s.far2 = 0; s.side_p = 0; s.side_n = 0;
      }
      s_parent[r] = c < MAX_COMPONENTS ? -2 - c : -1;
    }
  }
  __syncthreads();
#pragma unroll
  for (int k = 0; k < RUNS_RUN_CAP / RUNS_THREADS; ++k) {
    const int r = tid + k * RUNS_THREADS;
    if (r < total && root[k] != r) s_parent[r] = s_parent[root[k]];
  }
  __syncthreads();
  // ---- hand-over to boundary_list_kernel: the code of every run and the first run of every entry
  for (int r = tid; r < total; r += RUNS_THREADS) run_code[(int64_t)f * RUNS_RUN_CAP + r] = s_parent[r];
  for (int e = tid; e < n; e += RUNS_THREADS) ent_base[(int64_t)f * RUNS_ENT_CAP + e] = s_base[e];
}

// joins: a run with the run to its left across an item boundary, and a run with the run above it - once per pair of runs (at
// the first column where both are dark), not once per pixel
__global__ void ccl_merge_kernel(int w, int h, AGT_WIN_ARGS, int* __restrict__ label, const uint32_t* __restrict__ mask, int64_t mask_stride,
                                 const int* __restrict__ n_entries, const int2* __restrict__ entries, const uint8_t* __restrict__ overflow) {
  if (!overflow[blockIdx.y]) return;
  int* L = label + (int64_t)blockIdx.y * w * h;
  const uint32_t* M = mask + blockIdx.y * mask_stride;
  const int2* E = entries + blockIdx.y * mask_stride;
  AGT_WARP_SETUP
  const int n = n_entries[f];
  for (int e = warp0 * 2; e < n; e += nwarps * 2) {
    Entry t[2];
    unsigned up[2], lw[2], ulw[2];
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      t[k] = load_entry(E, e + k, n, chunks, win.ww, lane);
      up[k] = t[k].y > 0 ? M[t[k].item - chunks] : 0u;
      lw[k] = t[k].ch > 0 ? M[t[k].item - 1] : 0u;
      ulw[k] = t[k].ch > 0 && t[k].y > 0 ? M[t[k].item - chunks - 1] : 0u;
    }
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      const unsigned m = t[k].m, left_m = (m << 1) | (lw[k] >> 31), left_u = (up[k] << 1) | (ulw[k] >> 31);
      const unsigned join_up = m & up[k] & ~(left_m & left_u);
      if (lane == 0 && (m & 1u) && (lw[k] >> 31)) ccl_union(L, t[k].i, t[k].i - 1);
      if (join_up >> lane & 1u) ccl_union(L, t[k].i, t[k].i - win.ww);
    }
  }
}

// area of every component of an overflowing frame, at its root: each run adds its length (the counter of a root is the one
// ccl_runs_kernel cleared at the run's first pixel; it lives in the boundary list's scratch, which nobody uses before
// boundary_list_kernel)
__global__ void ccl_area_kernel(int w, int h, AGT_WIN_ARGS, const int* __restrict__ label, const int* __restrict__ n_entries,
                                const int2* __restrict__ entries, int64_t mask_stride, const uint8_t* __restrict__ overflow,
                                int2* __restrict__ area_scratch) {
  if (!overflow[blockIdx.y]) return;
  const int* L = label + (int64_t)blockIdx.y * w * h;
  int* A = reinterpret_cast<int*>(area_scratch + (int64_t)blockIdx.y * w * h);
  const int2* E = entries + blockIdx.y * mask_stride;
  AGT_WARP_SETUP
  const int n = n_entries[f];
  for (int e = warp0; e < n; e += nwarps) {
    const Entry t = load_entry(E, e, n, chunks, win.ww, lane);
    if (((t.m & ~(t.m << 1)) >> lane) & 1u) {
      const unsigned rest = ~(t.m >> lane);
      atomicAdd(&A[ccl_find(L, t.i)], rest == 0u ? 32 : __ffs(rest) - 1);
    }
  }
}

// every dark pixel is pointed at its root, and a root gets a component number on the spot: L[root] = -2 - number (numbers
// beyond MAX_COMPONENTS are dropped: L[root] = -1 marks nothing; as in ccl_runs_kernel, only roots of area >= 48 are numbered).
// A thread that walks through a root another thread has just numbered sees a negative value there and stops: ccl_find.
__global__ void ccl_flatten_number_kernel(int w, int h, AGT_WIN_ARGS, int* __restrict__ label, const int* __restrict__ n_entries,
                                          const int2* __restrict__ entries, int64_t mask_stride, int* __restrict__ n_comp, CompStats* __restrict__ stats,
                                          const uint8_t* __restrict__ overflow, const int2* __restrict__ area_scratch) {
  if (!overflow[blockIdx.y]) return;
  int* L = label + (int64_t)blockIdx.y * w * h;
  const int* A = reinterpret_cast<const int*>(area_scratch + (int64_t)blockIdx.y * w * h);
  const int2* E = entries + blockIdx.y * mask_stride;
  AGT_WARP_SETUP
  const int n = n_entries[f];
  for (int e = warp0 * 2; e < n; e += nwarps * 2) {
    Entry t[2];
    int me[2];
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      t[k] = load_entry(E, e + k, n, chunks, win.ww, lane);
      me[k] = t[k].dark ? L[t[k].i] : -1;
    }
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      if (me[k] < 0) continue;
      const int i = t[k].i;
      if (me[k] == i) {
        const int c = A[i] >= 48 ? atomicAdd(&n_comp[f], 1) : MAX_COMPONENTS;
        if (c < MAX_COMPONENTS) {
          CompStats& s = stats[(int64_t)f * MAX_COMPONENTS + c];
          s.area = 0; s.x0 = win.ww; s.y0 = win.hh; s.x1 = -1; s.y1 = -1; s.sx = 0; s.sy = 0; s.far0 = 0; s.far2 = 0; s.side_p = 0; s.side_n = 0;
        }
        L[i] = c < MAX_COMPONENTS ? -2 - c : -1;
      } else {
        const int r = ccl_find(L, me[k]);
        if (r != me[k]) L[i] = r;
      }
    }
  }
}

// after ccl_flatten_number_kernel: a root holds its code, every other dark pixel the index of its root
__device__ __forceinline__ int comp_of(const int* L, int l) {
  if (l == -1) return -1;
  if (l <= -2) return -2 - l;                   // a root
  const int r = L[l];
  return r <= -2 ? -2 - r : -1;
}
// the code of a run in ccl_runs_kernel's table
__device__ __forceinline__ int comp_code(int l) { return l <= -2 ? -2 - l : -1; }

// The quadrilateral of a component comes from its boundary pixels (a dark pixel with a background pixel, or the edge of the
// window, next to it) in three passes - 0: farthest from the centroid (c0); 1: farthest from c0 (c2); 2: farthest from the line
// c0 c2 on each side.  boundary_list_kernel (a thread per entry, mask arithmetic only) lists the boundary pixels of a frame;
// the three passes run a thread per listed pixel.  The same kernel adds up each component's statistics run by run, on either
// union-find path (the run's code: from ccl_runs_kernel's table, or - frames that overflowed it - from the pixel labels).
__global__ void boundary_list_kernel(int w, int h, AGT_WIN_ARGS, const int* __restrict__ label, const uint32_t* __restrict__ mask, int64_t mask_stride,
                                     const int* __restrict__ n_entries, const int2* __restrict__ entries, const uint8_t* __restrict__ overflow,
                                     const int* __restrict__ run_code, const int* __restrict__ ent_base, CompStats* __restrict__ stats,
                                     int* __restrict__ n_list, int2* __restrict__ list) {
  const int f = blockIdx.y;
  const Win win = frame_window(rects, rect_stride, f, w, h);
  const int chunks = (win.ww + 31) >> 5, n = n_entries[f];
  const bool by_label = overflow[f] != 0;
  const int* L = label + (int64_t)f * w * h;
  const uint32_t* M = mask + f * mask_stride;
  const int2* E = entries + f * mask_stride;
  const int* code = run_code + (int64_t)f * RUNS_RUN_CAP;
  int2* P = list + (int64_t)f * w * h;
  const int lane = threadIdx.x & 31;
  for (int e0 = blockIdx.x * blockDim.x + threadIdx.x - lane; e0 < n; e0 += gridDim.x * blockDim.x) {      // (uniform across a warp)
    const int e = e0 + lane;
    const bool act = e < n;
    const int2 v = act ? E[e] : make_int2(0, 0);
    const int item = v.x, y = item / chunks, ch = item - y * chunks;
    const unsigned m = (unsigned)v.y;
    const unsigned up = act && y > 0 ? M[item - chunks] : 0u, dn = act && y < win.hh - 1 ? M[item + chunks] : 0u;
    const unsigned lw = act && ch > 0 ? M[item - 1] : 0u, rw = act && ch < chunks - 1 ? M[item + 1] : 0u;
    const int base = by_label || !act ? 0 : ent_base[(int64_t)f * RUNS_ENT_CAP + e];
    const int xb = ch * 32, i0 = y * win.ww + xb;
    // (a neighbour outside the window reads as background: the edge of the window is a boundary)
    const unsigned bm = m & ~(((m << 1) | (lw >> 31)) & ((m >> 1) | (rw << 31)) & up & dn);
    // room in the list for the boundary pixels of the warp's 32 items by one addition
    const int cnt = __popc(bm);
    int incl = cnt;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int u = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += u; }
    const int total = __shfl_sync(0xffffffffu, incl, 31);
    int pos = lane == 0 && total > 0 ? atomicAdd(&n_list[f], total) : 0;
    pos = __shfl_sync(0xffffffffu, pos, 0) + incl - cnt;
    // run by run: the component's statistics (length, coordinate sums, extent) and the boundary pixels of the run
    // (adding the statistics up in ccl_runs_kernel with shared-memory atomics instead was measured: that kernel 20 -> 47 us, this
    // one 30 -> 19 us per 64 windows - one CTA's atomics on a border's seven words are slower than the whole grid's at the L2)
    unsigned mm = m;
    int r = 0;
    while (mm) {
      const int a = __ffs(mm) - 1;
      const unsigned t = mm >> a;
      const int len = t == 0xffffffffu ? 32 : __ffs(~t) - 1;
      const unsigned bits = (len == 32 ? 0xffffffffu : (1u << len) - 1u) << a;
      mm &= ~bits;
      const int c = by_label ? comp_of(L, L[i0 + a]) : comp_code(code[base + r++]);
      if (c >= 0) {
        CompStats& st = stats[(int64_t)f * MAX_COMPONENTS + c];
        const int xa = xb + a;
        atomicAdd(&st.area, len);
        atomicAdd(&st.sx, (unsigned long long)(len * xa + len * (len - 1) / 2)); atomicAdd(&st.sy, (unsigned long long)y * len);
        // the extent only ever grows: look first (past the L1), most runs lie inside what is there already
        if (xa < __ldcg(&st.x0)) atomicMin(&st.x0, xa);
        if (xa + len - 1 > __ldcg(&st.x1)) atomicMax(&st.x1, xa + len - 1);
        if (y < __ldcg(&st.y0)) atomicMin(&st.y0, y);
        if (y > __ldcg(&st.y1)) atomicMax(&st.y1, y);
      }
      unsigned bb = bm & bits;
      while (bb) { const int b = __ffs(bb) - 1; bb &= bb - 1; P[pos++] = make_int2(i0 + b, c); }
    }
  }
}

// one pass of the quadrilateral fit over boundary pixels e0, e0 + stride, ... of frame f (pass 0: farthest from the centroid,
// 1: farthest from that pixel, 2: farthest from the line through the two, on either side).  The keys of the previous pass are
// read past the L1 (they were written by atomics)
__device__ __forceinline__ void far_pass(int f, int ww, const int2* __restrict__ P, int n, CompStats* __restrict__ stats, int pass, int e0, int stride) {
  for (int e = e0; e < n; e += stride) {
    const int2 ic = P[e];
    const int i = ic.x, c = ic.y;
    if (c < 0) continue;
    CompStats& s = stats[(int64_t)f * MAX_COMPONENTS + c];
    const int area = s.area;
    if (area < 48) continue;
    const int y = i / ww, x = i - y * ww;
    if (pass == 0) {
      const float cx = (float)((double)s.sx / area), cy = (float)((double)s.sy / area);
      atomicMax(&s.far0, far_key((x - cx) * (x - cx) + (y - cy) * (y - cy), i));
    } else if (pass == 1) {
      const int p0 = (int)(__ldcg(&s.far0) & 0xffffffffu), x0 = p0 % ww, y0 = p0 / ww;
      atomicMax(&s.far2, far_key((float)((x - x0) * (x - x0) + (y - y0) * (y - y0)), i));
    } else {
      const int p0 = (int)(__ldcg(&s.far0) & 0xffffffffu), p2 = (int)(__ldcg(&s.far2) & 0xffffffffu);
      const int x0 = p0 % ww, y0 = p0 / ww, x2 = p2 % ww, y2 = p2 / ww;
      const float d = (float)((x2 - x0) * (y - y0) - (y2 - y0) * (x - x0));       // twice the signed area of (c0, c2, p)
      if (d > 0.f) atomicMax(&s.side_p, far_key(d, i));
      else if (d < 0.f) atomicMax(&s.side_n, far_key(-d, i));
    }
  }
}

__global__ void comp_far_kernel(int w, int h, AGT_WIN_ARGS, const int* __restrict__ n_list, const int2* __restrict__ list,
                                CompStats* __restrict__ stats, int pass) {
  const int f = blockIdx.y;
  const Win win = frame_window(rects, rect_stride, f, w, h);
  far_pass(f, win.ww, list + (int64_t)f * w * h, n_list[f], stats, pass, blockIdx.x * blockDim.x + threadIdx.x, gridDim.x * blockDim.x);
}

// component c of frame f: quadrilateral test, clockwise-on-screen order, emit (frame coordinates)
__device__ __forceinline__ void emit_quad(int f, int c, const Win win, const CompStats* __restrict__ stats, float* __restrict__ quads,
                                          uint8_t* __restrict__ quad_valid, uint8_t* __restrict__ quad_win, int* __restrict__ n_quads,
                                          int max_quads, int refine_win) {
  const CompStats* sp = stats + (int64_t)f * MAX_COMPONENTS + c;
  const int s_area = sp->area;
  if (s_area < 48 || sp->x0 <= 0 || sp->y0 <= 0 || sp->x1 >= win.ww - 1 || sp->y1 >= win.hh - 1) return;      // too small / cut by the window
  const unsigned long long far0 = __ldcg(&sp->far0), far2 = __ldcg(&sp->far2), side_p = __ldcg(&sp->side_p), side_n = __ldcg(&sp->side_n);
  if (far0 == 0 || far2 == 0 || side_p == 0 || side_n == 0) return;
  const int p[4] = {(int)(far0 & 0xffffffffu), (int)(side_p & 0xffffffffu), (int)(far2 & 0xffffffffu), (int)(side_n & 0xffffffffu)};
  float qx[4], qy[4];
  for (int k = 0; k < 4; ++k) { qx[k] = (float)(p[k] % win.ww); qy[k] = (float)(p[k] / win.ww); }
  // the component is the tag's black border plus the dark cells attached to it: between ~30 % (border alone) and 100 % of its quad
  float area2 = 0.f;
  for (int k = 0; k < 4; ++k) area2 += qx[k] * qy[(k + 1) & 3] - qx[(k + 1) & 3] * qy[k];
  const float qa = 0.5f * fabsf(area2);
  if (qa < 64.f || (float)s_area < 0.25f * qa || (float)s_area > 1.15f * qa) return;
  // shortest side at least 6 px, and not a sliver
  float smin = 1e30f, smax = 0.f, mean_side = 0.f;
  for (int k = 0; k < 4; ++k) {
    const float dx = qx[(k + 1) & 3] - qx[k], dy = qy[(k + 1) & 3] - qy[k], l = sqrtf(dx * dx + dy * dy);
    smin = fminf(smin, l); smax = fmaxf(smax, l); mean_side += 0.25f * l;
  }
  if (smin < 6.f || smin < 0.08f * smax) return;
  const int slot = atomicAdd(&n_quads[f], 1);
  if (slot >= max_quads) return;
  float* q = quads + ((int64_t)f * max_quads + slot) * 8;
  // clockwise on the screen (y down) = positive shoelace sum: the reference's order BL, TL, TR, BR runs that way
  const bool cw = area2 > 0.f;
  const float cx = (float)((double)sp->sx / s_area), cy = (float)((double)sp->sy / s_area);
  for (int k = 0; k < 4; ++k) {
    const int j = cw ? k : (4 - k) & 3;
    // the corner pixels are dark pixels just inside the tag: move half a pixel outwards from the centroid
    const float dx = qx[j] - cx, dy = qy[j] - cy, l = fmaxf(sqrtf(dx * dx + dy * dy), 1e-3f);
    q[2 * k] = (float)win.x0 + qx[j] + 0.5f * dx / l; q[2 * k + 1] = (float)win.y0 + qy[j] + 0.5f * dy / l;
  }
  quad_valid[(int64_t)f * max_quads + slot] = 1;
  // corner-refinement window: half a tag cell (a cell = an eighth of the side), so that the window of a small tag does not reach
  // the corners of its inner cells (the rule of OpenCV's ArUco detector, relativeCornerRefinmentWinSize), at most refine_win
  const int cwin = min(max((int)(0.5f * mean_side / 8.f + 0.5f), 2), max(refine_win, 1));
  for (int k = 0; k < 4; ++k) quad_win[((int64_t)f * max_quads + slot) * 4 + k] = (uint8_t)cwin;
}

// one thread per component; the first thread of a frame also clears the frame's tag counter (decode_tags_kernel counts into it)
__global__ void quad_emit_kernel(int w, int h, AGT_WIN_ARGS, const int* __restrict__ n_comp, const CompStats* __restrict__ stats,
                                 float* __restrict__ quads, uint8_t* __restrict__ quad_valid, uint8_t* __restrict__ quad_win, int* __restrict__ n_quads,
                                 int max_quads, int refine_win, int32_t* __restrict__ out_n) {
  const int f = blockIdx.y, c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c == 0 && out_n != nullptr) out_n[f] = 0;
  if (c >= min(n_comp[f], MAX_COMPONENTS)) return;
  emit_quad(f, c, frame_window(rects, rect_stride, f, w, h), stats, quads, quad_valid, quad_win, n_quads, max_quads, refine_win);
}

// Batches: the three passes and the emission of a frame by one thread-block cluster - a cluster barrier between the passes
// instead of a kernel boundary (four launches of 6-8 us, most of it ramp, tail and the first dependent loads, for microseconds
// of work): 23.4 against 28 us per 64 windows.  Measured and dropped: one CTA per frame (33.6 us: too few threads for the work),
// the boundary list in the same cluster kernel with 512 threads per CTA (53 against 20 + 23 us).
constexpr int FIT_CLUSTER = 8, FIT_THREADS = 256;
__global__ void __launch_bounds__(FIT_THREADS)
quad_fit_cluster_kernel(int w, int h, AGT_WIN_ARGS, const int* __restrict__ n_list, const int2* __restrict__ list, const int* __restrict__ n_comp,
                        CompStats* __restrict__ stats, float* __restrict__ quads, uint8_t* __restrict__ quad_valid, uint8_t* __restrict__ quad_win,
                        int* __restrict__ n_quads, int max_quads, int refine_win, int32_t* __restrict__ out_n) {
  namespace cg = cooperative_groups;
  cg::cluster_group cluster = cg::this_cluster();
  const int f = blockIdx.x / FIT_CLUSTER, rank = blockIdx.x % FIT_CLUSTER, t = rank * FIT_THREADS + threadIdx.x;
  const Win win = frame_window(rects, rect_stride, f, w, h);
  const int2* P = list + (int64_t)f * w * h;
  const int n = n_list[f];
  if (t == 0 && out_n != nullptr) out_n[f] = 0;
  for (int pass = 0; pass < 3; ++pass) {
    far_pass(f, win.ww, P, n, stats, pass, t, FIT_CLUSTER * FIT_THREADS);
    __threadfence();
    cluster.sync();
  }
  const int nc = min(n_comp[f], MAX_COMPONENTS);
  for (int c = t; c < nc; c += FIT_CLUSTER * FIT_THREADS) emit_quad(f, c, win, stats, quads, quad_valid, quad_win, n_quads, max_quads, refine_win);
}

// warp per frame, lane per group position: the detection of that tag with the largest margin (a tag reported twice fills one slot)
__global__ void pack_detections_kernel(const int32_t* __restrict__ n_det, const int32_t* __restrict__ det_id, const float* __restrict__ det_corners,
                                       const float* __restrict__ det_margin, int max_tags, const int32_t* __restrict__ group_ids, int n_group,
                                       float min_margin, float* __restrict__ img_pts, uint8_t* __restrict__ valid, int32_t* __restrict__ n_tags,
                                       int32_t* __restrict__ n_unknown, int batch) {
  const int lane = threadIdx.x & 31;
  const int f = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (f >= batch) return;
  const int nd = min(n_det[f], max_tags);
  const int32_t* ids = det_id + (int64_t)f * max_tags;
  const float* mg = det_margin ? det_margin + (int64_t)f * max_tags : nullptr;
  int count = 0, matched = 0;
  for (int pos = lane; pos < n_group; pos += 32) {
    const int want = group_ids[pos];
    int best = -1;
    float best_m = 0.f, best_x = 0.f;
    for (int k = 0; k < nd; ++k) {
      if (ids[k] != want) continue;
      const float m = mg ? mg[k] : min_margin;
      if (!(m >= min_margin)) continue;                        // detect_pose.py:389: decision_margin < 50 is skipped
      ++matched;
      const float x = det_corners[((int64_t)f * max_tags + k) * 8];
      if (best < 0 || m > best_m || (m == best_m && x < best_x)) { best = k; best_m = m; best_x = x; }
    }
    float* o = img_pts + ((int64_t)f * n_group + pos) * 8;
    uint8_t* v = valid + ((int64_t)f * n_group + pos) * 4;
    if (best >= 0) {
      const float* c = det_corners + ((int64_t)f * max_tags + best) * 8;
      for (int j = 0; j < 8; ++j) o[j] = c[j];
      v[0] = v[1] = v[2] = v[3] = 1;
      ++count;
    } else {
      for (int j = 0; j < 8; ++j) o[j] = 0.f;
      v[0] = v[1] = v[2] = v[3] = 0;
    }
  }
  int kept = 0;                                                // detections that pass the margin filter, whatever their id
  for (int k = lane; k < nd; k += 32) kept += (!mg || mg[k] >= min_margin) ? 1 : 0;
  count = __reduce_add_sync(0xffffffffu, count); matched = __reduce_add_sync(0xffffffffu, matched); kept = __reduce_add_sync(0xffffffffu, kept);
  if (lane == 0) {
    n_tags[f] = count;
    if (n_unknown) n_unknown[f] = kept - matched;              // ids outside the group: the reference raises KeyError on them
  }
}

}  // namespace

int agt_corner_subpix_windows(agt_ctx* ctx, const uint8_t* d_gray, int w, int h, int64_t pitch, int64_t stride, const float* d_pts,
                              const uint8_t* d_valid, const uint8_t* d_win, float* d_out, int batch, int n_pts, int win, int max_iters,
                              double eps);

// the detector's scratch: the pixel labels in slot 0, everything else in slot 1 (byte offsets into it)
struct TagScratch {
  int* label;
  uint8_t* ws;
  size_t o_stats, o_lohi, o_ncomp, o_nlist, o_nent, o_over, o_nquads, o_qvalid, o_win, o_quads, o_refined, o_id, o_rot, o_ham, o_margin, o_list,
      o_mask, o_ent, o_pos, o_rcode, o_ebase, o_tiles, total;
};

// first half of the detector: threshold -> components -> farthest points -> quads (ws + o_quads, validity flags, refinement
// windows; per frame the number of components numbered, the union-find that ran and the number of quads found).  out_n
// (nullable): the detector's tag counters, cleared by the emission
static int find_quads(agt_ctx* ctx, const uint8_t* d_gray, int w, int h, int64_t pitch, int64_t stride, int batch, const int32_t* d_rects,
                      int rect_stride, int max_quads, int refine_win, int32_t* out_n, TagScratch& S) {
  const int64_t n = (int64_t)w * h, mask_stride = (int64_t)((w + 31) / 32) * h;
  const int64_t tile_stride = ((int64_t)((w + 31) / 32) * ((h + TILE - 1) / TILE) + 63) & ~(int64_t)63;
  // whole frames take the local white level, search windows one threshold each (agt_set_tag_threshold overrides)
  const bool local = ctx->tag_threshold == 2 || (ctx->tag_threshold == 0 && d_rects == nullptr);
  int rc;
  if ((rc = agt_scratch(ctx, 0, sizeof(int) * (size_t)n * batch, reinterpret_cast<void**>(&S.label)))) return rc;
  S.o_stats = 0; S.o_lohi = S.o_stats + sizeof(CompStats) * (size_t)MAX_COMPONENTS * batch; S.o_ncomp = S.o_lohi + sizeof(int) * 2 * batch;
  S.o_nlist = S.o_ncomp + sizeof(int) * batch; S.o_nent = S.o_nlist + sizeof(int) * batch; S.o_over = S.o_nent + sizeof(int) * batch;
  S.o_nquads = (S.o_over + (size_t)batch + 3) & ~(size_t)3;
  S.o_qvalid = S.o_nquads + sizeof(int) * batch; S.o_win = S.o_qvalid + (size_t)max_quads * batch;             // everything up to here starts as zero
  S.o_quads = (S.o_win + 4 * (size_t)max_quads * batch + 63) & ~(size_t)63; S.o_refined = S.o_quads + sizeof(float) * 8 * (size_t)max_quads * batch;
  S.o_id = (S.o_refined + sizeof(float) * 8 * (size_t)max_quads * batch + 63) & ~(size_t)63;
  S.o_rot = S.o_id + sizeof(int32_t) * (size_t)max_quads * batch; S.o_ham = S.o_rot + (size_t)max_quads * batch;
  S.o_margin = (S.o_ham + (size_t)max_quads * batch + 63) & ~(size_t)63;
  S.o_list = (S.o_margin + sizeof(float) * (size_t)max_quads * batch + 63) & ~(size_t)63; S.o_mask = S.o_list + sizeof(int2) * (size_t)n * batch;
  S.o_ent = (S.o_mask + sizeof(uint32_t) * (size_t)mask_stride * batch + 63) & ~(size_t)63; S.o_pos = S.o_ent + sizeof(int2) * (size_t)mask_stride * batch;
  S.o_rcode = S.o_pos + sizeof(int) * (size_t)mask_stride * batch; S.o_ebase = S.o_rcode + sizeof(int) * (size_t)RUNS_RUN_CAP * batch;
  S.o_tiles = S.o_ebase + sizeof(int) * (size_t)RUNS_ENT_CAP * batch; S.total = S.o_tiles + (size_t)tile_stride * batch;
  if ((rc = agt_scratch(ctx, 1, S.total, reinterpret_cast<void**>(&S.ws)))) return rc;
  uint8_t* ws = S.ws;
  int* label = S.label;
  CompStats* stats = reinterpret_cast<CompStats*>(ws + S.o_stats);
  int *lohi = reinterpret_cast<int*>(ws + S.o_lohi), *ncomp = reinterpret_cast<int*>(ws + S.o_ncomp), *nlist = reinterpret_cast<int*>(ws + S.o_nlist),
      *nent = reinterpret_cast<int*>(ws + S.o_nent), *nquads = reinterpret_cast<int*>(ws + S.o_nquads);
  float* quads = reinterpret_cast<float*>(ws + S.o_quads);
  uint8_t* qvalid = ws + S.o_qvalid;
  int2* far_list = reinterpret_cast<int2*>(ws + S.o_list);
  int2* entries = reinterpret_cast<int2*>(ws + S.o_ent);
  uint32_t* mask = reinterpret_cast<uint32_t*>(ws + S.o_mask);
  int* entry_of = reinterpret_cast<int*>(ws + S.o_pos);
  uint8_t* overflow = ws + S.o_over;
  int *run_code = reinterpret_cast<int*>(ws + S.o_rcode), *ent_base = reinterpret_cast<int*>(ws + S.o_ebase);
  cudaStream_t st = ctx->stream;
  // one memset: darkest / brightest pixel (stored so that both start as 0), counters, overflow flags, validity flags and
  // refinement windows of the quads; the tag counters are cleared by the quad emission
  AGT_CUDA(ctx, cudaMemsetAsync(ws + S.o_lohi, 0, S.o_quads - S.o_lohi, st));
  // grid-stride over the pixels of each frame's window; with windows (usually a few percent of the frame) a smaller grid per frame
  // (whole frames: 32 CTAs per SM over the batch - a grid sized for one frame, times 64 frames, spent its time launching CTAs
  // that had nothing to do: 174 + 188 us for min/max + threshold of 64 1080p frames)
  const int64_t per_frame = std::max<int64_t>(16, (int64_t)(d_rects ? 8 : 32) * ctx->sm_count / batch);
  const dim3 grid((unsigned)std::min<int64_t>((n + 255) / 256, per_frame), (unsigned)batch);
  // the passes over the list of non-empty items / boundary pixels: sized for the dark part of a frame, whatever the window
  const dim3 grid_ne((unsigned)std::min<int64_t>((n + 255) / 256, std::max<int64_t>(16, (int64_t)8 * ctx->sm_count / batch)), (unsigned)batch);
  // (both passes of a frame by one CTA of 1024 threads - one launch, tile maxima in shared memory, the second read from the L2 -
  // measured slower: 48 against 13 + 21 us per 64 windows, 293 against 57 + 80 us per 64 whole frames; the threshold pass is
  // instruction work - dark bits, runs, first labels - that one SM per frame does not get through)
  uint8_t* tiles = local ? ws + S.o_tiles : nullptr;
  if (local) tile_max_kernel<<<grid, 256, 0, st>>>(d_gray, w, h, pitch, stride, d_rects, rect_stride, lohi, tiles, tile_stride);
  else frame_minmax_kernel<<<grid, 256, 0, st>>>(d_gray, w, h, pitch, stride, d_rects, rect_stride, lohi);
  ccl_init_kernel<<<grid, 256, 0, st>>>(d_gray, w, h, pitch, stride, d_rects, rect_stride, lohi, tiles, tile_stride, mask, mask_stride, nent, entries,
                                       entry_of);
  ccl_runs_kernel<<<(unsigned)batch, RUNS_THREADS, 0, st>>>(w, h, d_rects, rect_stride, mask, mask_stride, nent, entries, entry_of, ncomp, stats,
                                                           overflow, run_code, ent_base, label, far_list);
  ccl_merge_kernel<<<grid_ne, 256, 0, st>>>(w, h, d_rects, rect_stride, label, mask, mask_stride, nent, entries, overflow);
  ccl_area_kernel<<<grid_ne, 256, 0, st>>>(w, h, d_rects, rect_stride, label, nent, entries, mask_stride, overflow, far_list);
  ccl_flatten_number_kernel<<<grid_ne, 256, 0, st>>>(w, h, d_rects, rect_stride, label, nent, entries, mask_stride, ncomp, stats, overflow, far_list);
  boundary_list_kernel<<<grid_ne, 256, 0, st>>>(w, h, d_rects, rect_stride, label, mask, mask_stride, nent, entries, overflow, run_code, ent_base, stats,
                                                nlist, far_list);
  if (batch >= 8) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)batch * FIT_CLUSTER);
    cfg.blockDim = dim3(FIT_THREADS);
    cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = FIT_CLUSTER; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    const int* c_nlist = nlist; const int2* c_list = far_list; const int* c_ncomp = ncomp;
    uint8_t* qwin = ws + S.o_win;
    const cudaError_t e = cudaLaunchKernelEx(&cfg, quad_fit_cluster_kernel, w, h, d_rects, rect_stride, c_nlist, c_list, c_ncomp, stats, quads,
                                             qvalid, qwin, nquads, max_quads, refine_win, out_n);
    if (e != cudaSuccess) AGT_FAIL(ctx, AGT_ERR_CUDA, "agt_detect_tags: cluster launch failed: %s", cudaGetErrorString(e));
  } else {
    for (int pass = 0; pass < 3; ++pass) comp_far_kernel<<<grid_ne, 256, 0, st>>>(w, h, d_rects, rect_stride, nlist, far_list, stats, pass);
    quad_emit_kernel<<<dim3(MAX_COMPONENTS / 128, (unsigned)batch), 128, 0, st>>>(w, h, d_rects, rect_stride, ncomp, stats, quads, qvalid,
                                                                                     ws + S.o_win, nquads, max_quads, refine_win, out_n);
  }
  AGT_LAUNCH_CHECK(ctx);
  return AGT_OK;
}

static bool tag_args_ok(const uint8_t* d_gray, int w, int h, int64_t pitch, int batch, int refine_win) {
  return d_gray && batch > 0 && batch <= 65535 && w >= 16 && h >= 16 && pitch >= w && (int64_t)w * h <= 0x7fffffffLL && refine_win >= 0 &&
         refine_win <= 7;
}

extern "C" int agt_tag_quads(agt_ctx* ctx, const uint8_t* d_gray, int w, int h, int64_t pitch, int64_t stride, int batch, const int32_t* d_rects,
                             int rect_stride, int max_quads, int refine_win, int32_t* d_n_comp, uint8_t* d_overflow, int32_t* d_n_quads,
                             float* d_quads, uint8_t* d_quad_win) {
  if (!ctx) return AGT_ERR_INVALID;
  if (d_rects != nullptr && rect_stride < 4) AGT_FAIL(ctx, AGT_ERR_INVALID, "agt_tag_quads: rect_stride < 4");
  if (batch == 0) return AGT_OK;
  if (!tag_args_ok(d_gray, w, h, pitch, batch, refine_win) || max_quads < 1 || max_quads > MAX_COMPONENTS || !d_n_comp || !d_overflow || !d_n_quads ||
      !d_quads || !d_quad_win)
    AGT_FAIL(ctx, AGT_ERR_INVALID, "agt_tag_quads: bad arguments");
  TagScratch S;
  int rc;
  if ((rc = find_quads(ctx, d_gray, w, h, pitch, stride, batch, d_rects, rect_stride, max_quads, refine_win, nullptr, S))) return rc;
  cudaStream_t st = ctx->stream;
  AGT_CUDA(ctx, cudaMemcpyAsync(d_n_comp, S.ws + S.o_ncomp, sizeof(int32_t) * (size_t)batch, cudaMemcpyDeviceToDevice, st));
  AGT_CUDA(ctx, cudaMemcpyAsync(d_overflow, S.ws + S.o_over, (size_t)batch, cudaMemcpyDeviceToDevice, st));
  AGT_CUDA(ctx, cudaMemcpyAsync(d_n_quads, S.ws + S.o_nquads, sizeof(int32_t) * (size_t)batch, cudaMemcpyDeviceToDevice, st));
  AGT_CUDA(ctx, cudaMemcpyAsync(d_quads, S.ws + S.o_quads, sizeof(float) * 8 * (size_t)max_quads * batch, cudaMemcpyDeviceToDevice, st));
  // (the detector keeps the window once per corner)
  AGT_CUDA(ctx, cudaMemcpy2DAsync(d_quad_win, 1, S.ws + S.o_win, 4, 1, (size_t)max_quads * batch, cudaMemcpyDeviceToDevice, st));
  return AGT_OK;
}

extern "C" int agt_detect_tags_roi(agt_ctx* ctx, const uint8_t* d_gray, int w, int h, int64_t pitch, int64_t stride, int batch,
                                   const int32_t* d_rects, int rect_stride, int max_tags, int max_hamming, int refine_win, int32_t* d_n_tags,
                                   int32_t* d_ids, float* d_corners, float* d_margin, uint8_t* d_hamming) {
  if (!ctx) return AGT_ERR_INVALID;
  if (d_rects != nullptr && rect_stride < 4) AGT_FAIL(ctx, AGT_ERR_INVALID, "agt_detect_tags_roi: rect_stride < 4");
  if (batch == 0) return AGT_OK;
  if (!ctx->d_tag_codes) AGT_FAIL(ctx, AGT_ERR_NOT_READY, "agt_detect_tags: call agt_set_tag_family first");
  if (!tag_args_ok(d_gray, w, h, pitch, batch, refine_win) || !d_n_tags || !d_ids || !d_corners || max_tags < 1 || max_tags > 1024)
    AGT_FAIL(ctx, AGT_ERR_INVALID, "agt_detect_tags: bad arguments");
  const int max_quads = 4 * max_tags < 64 ? 64 : 4 * max_tags;
  TagScratch S;
  int rc;
  if ((rc = find_quads(ctx, d_gray, w, h, pitch, stride, batch, d_rects, rect_stride, max_quads, refine_win, d_n_tags, S))) return rc;
  uint8_t* ws = S.ws;
  const float* use = reinterpret_cast<const float*>(ws + S.o_quads);
  if (refine_win > 0) {
    // only the corners of emitted quads (the validity flag of a quad, four times), each with its own window
    float* refined = reinterpret_cast<float*>(ws + S.o_refined);
    if ((rc = agt_corner_subpix_windows(ctx, d_gray, w, h, pitch, stride, use, ws + S.o_win, ws + S.o_win, refined, batch, 4 * max_quads,
                                        refine_win, TAG_SUBPIX_ITERS, 1e-3)))
      return rc;
    use = refined;
  }
  // identification; the quads that decode go straight to the caller's list (no collection pass)
  if ((rc = decode_tags(ctx, d_gray, w, h, pitch, stride, use, ws + S.o_qvalid, reinterpret_cast<int32_t*>(ws + S.o_id), ws + S.o_rot, ws + S.o_ham,
                        reinterpret_cast<float*>(ws + S.o_margin), batch, max_quads, max_hamming,
                        TagSink{d_n_tags, d_ids, d_corners, d_margin, d_hamming, max_tags})))
    return rc;
  AGT_LAUNCH_CHECK(ctx);
  return AGT_OK;
}

extern "C" int agt_detect_tags(agt_ctx* ctx, const uint8_t* d_gray, int w, int h, int64_t pitch, int64_t stride, int batch, int max_tags,
                               int max_hamming, int refine_win, int32_t* d_n_tags, int32_t* d_ids, float* d_corners, float* d_margin,
                               uint8_t* d_hamming) {
  return agt_detect_tags_roi(ctx, d_gray, w, h, pitch, stride, batch, nullptr, 0, max_tags, max_hamming, refine_win, d_n_tags, d_ids, d_corners,
                             d_margin, d_hamming);
}

extern "C" int agt_pack_detections(agt_ctx* ctx, const int32_t* d_n_det, const int32_t* d_det_ids, const float* d_det_corners,
                                   const float* d_det_margin, int max_tags, const int32_t* d_group_ids, int n_group, float min_margin,
                                   float* d_img_pts, uint8_t* d_valid, int32_t* d_n_tags, int32_t* d_n_unknown, int batch) {
  if (!ctx) return AGT_ERR_INVALID;
  if (batch == 0) return AGT_OK;
  if (!d_n_det || !d_det_ids || !d_det_corners || !d_group_ids || !d_img_pts || !d_valid || !d_n_tags || batch < 0 || max_tags < 1 ||
      n_group < 1 || n_group > 4096)
    AGT_FAIL(ctx, AGT_ERR_INVALID, "agt_pack_detections: bad arguments");
  pack_detections_kernel<<<(unsigned)((batch + 3) / 4), 128, 0, ctx->stream>>>(d_n_det, d_det_ids, d_det_corners, d_det_margin, max_tags,
                                                                              d_group_ids, n_group, min_margin, d_img_pts, d_valid, d_n_tags,
                                                                              d_n_unknown, batch);
  AGT_LAUNCH_CHECK(ctx);
  return AGT_OK;
}

extern "C" int agt_detect_tags_host(agt_ctx* ctx, const uint8_t* h_gray, int w, int h, int max_tags, int max_hamming, int refine_win,
                                    int32_t* h_n_tags, int32_t* h_ids, float* h_corners, float* h_margin, uint8_t* h_hamming) {
  if (!ctx) return AGT_ERR_INVALID;
  if (!h_gray || !h_n_tags || !h_ids || !h_corners || w < 16 || h < 16 || max_tags < 1 || max_tags > 1024)
    AGT_FAIL(ctx, AGT_ERR_INVALID, "agt_detect_tags_host: bad arguments");
  AGT_CUDA(ctx, cudaSetDevice(ctx->device));
  uint8_t *dimg, *dout;
  int rc;
  const size_t img_bytes = (size_t)w * h;
  const size_t o_n = 0, o_id = 64, o_c = o_id + sizeof(int32_t) * (size_t)max_tags, o_m = o_c + sizeof(float) * 8 * (size_t)max_tags,
               o_h = o_m + sizeof(float) * (size_t)max_tags, total = o_h + (size_t)max_tags;
  if ((rc = agt_scratch(ctx, 2, img_bytes, reinterpret_cast<void**>(&dimg)))) return rc;
  if ((rc = agt_scratch(ctx, 3, total, reinterpret_cast<void**>(&dout)))) return rc;
  cudaStream_t st = ctx->stream;
  AGT_CUDA(ctx, cudaMemcpyAsync(dimg, h_gray, img_bytes, cudaMemcpyHostToDevice, st));
  if ((rc = agt_detect_tags(ctx, dimg, w, h, w, (int64_t)img_bytes, 1, max_tags, max_hamming, refine_win, reinterpret_cast<int32_t*>(dout + o_n),
                            reinterpret_cast<int32_t*>(dout + o_id), reinterpret_cast<float*>(dout + o_c), reinterpret_cast<float*>(dout + o_m),
                            dout + o_h)))
    return rc;
  AGT_CUDA(ctx, cudaMemcpyAsync(h_n_tags, dout + o_n, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  AGT_CUDA(ctx, cudaMemcpyAsync(h_ids, dout + o_id, sizeof(int32_t) * (size_t)max_tags, cudaMemcpyDeviceToHost, st));
  AGT_CUDA(ctx, cudaMemcpyAsync(h_corners, dout + o_c, sizeof(float) * 8 * (size_t)max_tags, cudaMemcpyDeviceToHost, st));
  if (h_margin) AGT_CUDA(ctx, cudaMemcpyAsync(h_margin, dout + o_m, sizeof(float) * (size_t)max_tags, cudaMemcpyDeviceToHost, st));
  if (h_hamming) AGT_CUDA(ctx, cudaMemcpyAsync(h_hamming, dout + o_h, (size_t)max_tags, cudaMemcpyDeviceToHost, st));
  AGT_CUDA(ctx, cudaStreamSynchronize(st));
  if (*h_n_tags > max_tags) *h_n_tags = max_tags;
  return AGT_OK;
}
