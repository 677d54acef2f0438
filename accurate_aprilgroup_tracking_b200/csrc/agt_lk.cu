// K2: pyramidal Lucas-Kanade corner tracking, one warp per tracked corner.
//
// The reference snapshot has no optical-flow code; the frozen semantics are
// cv::calcOpticalFlowPyrLK(prev, next, prevPts, None) with its defaults
// (SURVEY.md 8a row A4, 9.2; restated in oracle/lk_oracle.py:lk_np): 21x21
// window, fixed-point bilinear weights (W_BITS 14), int16 template (x32) and
// int16 interpolated Scharr derivatives, float 2x2 structure tensor with the
// minEig 1e-4 gate, <= 30 iterations, |delta|^2 <= 1e-4 stop and the
// oscillation rule.  Outside the image the intensity is BORDER_REFLECT_101 and
// the derivative is zero, exactly as OpenCV's padded pyramids behave.
//
// Per corner and level the warp stages the 24x24 u8 template footprint in shared
// memory, derives the 22x22 Scharr values from it (no gradient plane is ever
// materialised in HBM), builds the 21x21 template, reduces the structure tensor
// with warp shuffles, then iterates against a 32x32 u8 search region staged
// from the next image (re-staged only if the window drifts out of it).
//
// Bit parity with OpenCV.  cv::calcOpticalFlowPyrLK accumulates the structure tensor and the mismatch vector in
// float32, in the order of its 128-bit SIMD loop (oracle/lk_oracle.py:_tensor_sum_f32 / _mismatch_sum_f32 restate it
// and are bit-identical to cv2 on every corner tried): columns 0..15 of a row go to four float lanes (lane k adds
// columns k, k+4, k+8, k+12; for the mismatch vector the products of columns (k, k+4) are first added as integers),
// rows top to bottom, the lanes are reduced as (l0+l2)+(l1+l3); columns 16..20 are added one at a time into a scalar
// float, and the lane sum is added to that scalar last.  The products exceed 2^24, so every one of those additions
// rounds, and on ill-conditioned windows one rounding decides whether another iteration runs (0.05 px).  This kernel
// therefore forms the same integer products in parallel, converts them exactly like cvtdq2ps, and adds them up in
// that very order: the owners write the floats to shared memory chain by chain, ten lanes then run the ten dependent
// chains (8 x 42 additions, 2 x 105).  Points, status and error come out bit-identical to OpenCV.
#include "agt_common.cuh"

namespace {

constexpr int WIN = 21;
constexpr int PATCH = WIN + 3;             // 24: template footprint incl. bilinear + Scharr halo
constexpr int DER = WIN + 1;               // 22
constexpr int REG = 32;                    // staged search region: REG columns x REG_H rows
constexpr int REG_H = 30;
constexpr int REG_MARGIN = 5;              // window offset inside a freshly staged region (columns / rows)
constexpr int REG_MARGIN_Y = 4;
// Shared-memory rows of the two staged footprints hold the aligned 32-bit words that cover the footprint's columns (the
// footprint starts `x & 3` bytes into the row): 7 words for 24 columns, 9 for 32.  An odd number of words per row also
// spreads the rows of a window over all banks (rows of 8 words put every fourth row on the same banks).
constexpr int PATCH_PITCH = 28, REG_PITCH = 36;
constexpr int WARPS_PER_CTA = 7;          // 4 CTAs of 7 warps: 4 x (7 x 8176 + 1024 reserved) bytes of an SM's 228 KB
constexpr int W_BITS = 14;
constexpr int MAX_ITERS = 30;

// Window pixels per lane, in two runs of consecutive pixels of one row each ("segments"), so that the search loop reads
// every run with three aligned 32-bit loads per image row instead of one byte load per tap:
//   lanes 0..20  ("row lanes") : row = lane, columns 0..7 and 8..15 - the part OpenCV's SIMD loop handles
//   lanes 21..31 ("tail lanes"): rows 2(l-21), 2(l-21)+1, columns 16..20 - OpenCV's scalar tail
// (lane 31's second run would be row 21: it is disabled by zero derivatives; a tail lane computes eight pixels per run
// like a row lane and uses the first five).  The per-pixel template arrays are lane-interleaved so that no access has a
// bank conflict: dd holds (dx, dy) of two neighbouring pixels per int4, run s / pixel pair p of lane l at
// dd[s * DD_RUN + (p < 3 ? 32 p : 96) + l] (pairs 0..2 for all 32 lanes, pair 3 for the row lanes only); tmpl holds the
// eight int16 template values of run s of lane l in tmpl[s][l].
constexpr int SEG_LEN = 8;
constexpr int TAIL_LEN = 5;
constexpr int DD_RUN = 3 * 32 + WIN;                                  // 117 int4 per run index
constexpr int REG_BYTES = (REG_H * REG_PITCH + 12 + 15) & ~15;        // + the third word of a run in the last row
// float scratch of the ordered sums.  Search loop: 8 chains of 42 (x / y, lanes 0..3 of the SIMD loop: element 2 row + group)
// and 2 chains of 105 (the scalar tail: element 5 row + column - 16), padded with zeros to whole float4s.  Structure tensor
// (before the region is staged): 84 per lane chain, in two passes (A11 and A12; A22 and the three tails).
constexpr int CH_SIMD = 44, CH_TAIL = 108, CH_A = 4 * WIN, CH_ATAIL = 112;

struct __align__(16) WarpSmem {
  union {
    struct {
      __align__(16) short2 der[DER][DER];  // Scharr at (ix..ix+21, iy..iy+21); the search region below overlays it
      __align__(16) uint8_t patch[PATCH * PATCH_PITCH];   // prev level, origin (ix-1, iy-1) at byte `x offset` of row 0
    } t;
    struct {
      __align__(16) uint8_t px[REG_BYTES];                  // next level search region
      __align__(16) float simd[8][CH_SIMD];
      __align__(16) float tail[2][CH_TAIL];
    } region;
    struct { __align__(16) float simd[8][CH_A]; } a1;
    struct { __align__(16) float simd[4][CH_A]; __align__(16) float tail[3][CH_ATAIL]; } a2;
  } u;
  __align__(16) int4 dd[2 * DD_RUN];       // template derivative (dx, dy) of two pixels
  __align__(16) uint4 tmpl[2][32];         // template intensity * 32, eight int16 per run
  // region-of-interest pyramids only: exact part [x_lo, x_hi) x [y_lo, y_hi) of the current level of the next pyramid and
  // the "looked outside" flag, kept here rather than in registers that would be live across the search loop
  __align__(16) int win[4];
  int left;
};
static_assert(sizeof(WarpSmem) <= 8192, "4 CTAs of 7 warps per SM");

__device__ __forceinline__ void segment_of(int lane, int s, int& row, int& col) {
  if (lane < WIN) { row = lane; col = SEG_LEN * s; }
  else { row = 2 * (lane - WIN) + s; col = 2 * SEG_LEN; }
}

// One dependent float32 chain per lane: acc = (..((acc + p[0].x) + p[0].y) + ..) over N4 float4s, one rounding per
// addition.  Straight-line code (the callers branch once around a whole chain) so that the loads run ahead of the adds.
template <int N4>
__device__ __forceinline__ float ordered_sum(const float4* __restrict__ p, float acc) {
  // (a rolled loop of four float4s per trip - a third less code, the kernel stalls 1.4 warps per issue on instruction fetch -
  // measured 2 % slower than the unrolled chain: 8.45 against 8.29 ms per 8192 frame pairs)
#pragma unroll
  for (int i = 0; i < N4; ++i) {
    const float4 v = p[i];
    acc = __fadd_rn(__fadd_rn(__fadd_rn(__fadd_rn(acc, v.x), v.y), v.z), v.w);
  }
  return acc;
}
// v_reduce_sum of the four SIMD lane accumulators held by lanes base..base+3: (l0 + l2) + (l1 + l3), valid in lane base
__device__ __forceinline__ float reduce_lanes4(float acc) {
  const float s = __fadd_rn(acc, __shfl_down_sync(0xffffffffu, acc, 2));
  return __fadd_rn(s, __shfl_down_sync(0xffffffffu, s, 1));
}

// Exact warp-wide sum of one 32-bit integer per lane (the total needs more than 32 bits).  Five 64-bit shuffle steps; the
// warp-reduce unit (two REDUX.SUM on the 16-bit halves) was measured 4-14 % slower for the whole kernel
// (profiles/r01_lk_variants.log).
__device__ __forceinline__ long long warp_sum_wide(int v) { return agt_warp_sum((long long)v); }

struct Weights { int w00, w01, w10, w11; };

__device__ __forceinline__ Weights make_weights(float a, float b) {
  Weights w;
  float na = __fsub_rn(1.f, a), nb = __fsub_rn(1.f, b);
  w.w00 = __float2int_rn(__fmul_rn(__fmul_rn(na, nb), 16384.f));
  w.w01 = __float2int_rn(__fmul_rn(__fmul_rn(a, nb), 16384.f));
  w.w10 = __float2int_rn(__fmul_rn(__fmul_rn(na, b), 16384.f));
  w.w11 = (1 << W_BITS) - w.w00 - w.w01 - w.w10;
  return w;
}

__device__ __forceinline__ int descale(int v, int n) { return (v + (1 << (n - 1))) >> n; }

// BORDER_REFLECT_101 index: in range for every window that is not cut by the image border (no modulo then)
__device__ __forceinline__ int reflect_fast(int i, int n) { return (unsigned)i < (unsigned)n ? i : agt_reflect101(i, n); }

// acc + sum_k px.byte[k] (unsigned) * coef.byte[k] (signed)
__device__ __forceinline__ int dp4us(uint32_t px, int coef, int acc) {
  int d;
  asm("dp4a.u32.s32 %0, %1, %2, %3;" : "=r"(d) : "r"(px), "r"(coef), "r"(acc));
  return d;
}

// The 9 bytes of a run (columns col..col+8 of one staged row) as two words with the run's first byte in bits 0-7, plus
// the same shifted by one byte: pixel k of the run blends bytes (k, k+1) of two rows, i.e. one half of one of these
// words per row, which is exactly what dp2a multiplies by a pair of 16-bit weights.
struct Run { uint32_t e0, e1, o0, o1; };
__device__ __forceinline__ Run load_run(uint32_t smem_addr) {
  const uint32_t wa = smem_addr & ~3u, sh = (smem_addr & 3u) * 8u;
  uint32_t w0, w1, w2;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(w0) : "r"(wa));
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(w1) : "r"(wa + 4));
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(w2) : "r"(wa + 8));
  Run r;
  r.e0 = __funnelshift_r(w0, w1, sh);
  r.e1 = __funnelshift_r(w1, w2, sh);
  r.o0 = __funnelshift_r(r.e0, r.e1, 8);
  r.o1 = __funnelshift_r(r.e1, w2 >> sh, 8);
  return r;
}
// bilinear value * 32 of pixel k (0..7) of a run: (w00 p00 + w01 p01 + w10 p10 + w11 p11 + 2^8) >> 9, the same integer
// OpenCV computes; wt = w00 | w01 << 16, wb = w10 | w11 << 16
// d = c + a.lo16 * b.byte[0 | 2] + a.hi16 * b.byte[1 | 3] with SIGNED 16-bit weights and unsigned pixel bytes: the fourth
// bilinear weight, 2^14 - w00 - w01 - w10, is -1 when the three rounded ones add up to 2^14 + 1 (OpenCV multiplies signed
// int16 weights, pmaddwd); the all-unsigned dp2a read that as 65535 - the cause of round 1's rare 0.05 px outliers.
__device__ __forceinline__ int dp2a_lo_su(uint32_t w, uint32_t px, int c) {
  int d;
  asm("dp2a.lo.s32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(w), "r"(px), "r"(c));
  return d;
}
__device__ __forceinline__ int dp2a_hi_su(uint32_t w, uint32_t px, int c) {
  int d;
  asm("dp2a.hi.s32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(w), "r"(px), "r"(c));
  return d;
}
template <int K>
__device__ __forceinline__ int blend(const Run& t, const Run& b, uint32_t wt, uint32_t wb) {
  const uint32_t tw = (K & 1) ? (K < 4 ? t.o0 : t.o1) : (K < 4 ? t.e0 : t.e1);
  const uint32_t bw = (K & 1) ? (K < 4 ? b.o0 : b.o1) : (K < 4 ? b.e0 : b.e1);
  const int acc = (K & 2) ? dp2a_hi_su(wb, bw, dp2a_hi_su(wt, tw, 256)) : dp2a_lo_su(wb, bw, dp2a_lo_su(wt, tw, 256));
  return acc >> (W_BITS - 5);
}

// Stage the footprint [x0, x0 + W) x [y0, y0 + ROWS) of one level into shared memory and return the byte offset of
// column x0 inside a shared-memory row.  Footprints inside the image (4-byte aligned rows) travel as aligned words by
// cp.async: every request of the footprint is in flight at once and no register waits for it.  Footprints cut by the
// image border are gathered byte by byte with BORDER_REFLECT_101 (a lane per column).  The caller waits.
// the rare path (a footprint cut by the image border), kept out of line so that it does not sit in the instruction
// stream of every warp: the kernel is large and the warps of an SM are spread all over it
__device__ __noinline__ void stage_footprint_bytes(uint8_t* smem, const uint8_t* __restrict__ img, int cols, int rows, int64_t pitch,
                                                   int x0, int y0, int lane, int w, int n_rows, int spitch) {
  const int gx = reflect_fast(x0 + (lane < w ? lane : 0), cols);
  for (int r = 0; r < n_rows; ++r) {
    const int gy = reflect_fast(y0 + r, rows);
    if (lane < w) smem[r * spitch + lane] = __ldg(img + (int64_t)gy * pitch + gx);
  }
}

template <int W, int ROWS, int WORDS, int SPITCH>
__device__ __forceinline__ int stage_footprint(uint8_t* smem, const uint8_t* __restrict__ img, int cols, int rows, int64_t pitch,
                                               int x0, int y0, int lane) {
  static_assert((WORDS == 9 || WORDS == 7) && WORDS * 4 == SPITCH && WORDS * 4 >= W + 3, "row of aligned words");
  if (x0 >= 0 && y0 >= 0 && x0 + W <= cols && y0 + ROWS <= rows && ((pitch | reinterpret_cast<uintptr_t>(img)) & 3) == 0) {
    const int xa = x0 & ~3, nw = ((x0 + W - 1) >> 2) - (x0 >> 2) + 1;
    const uint32_t sa = (uint32_t)__cvta_generic_to_shared(smem);
    const uint8_t* src = img + (int64_t)y0 * pitch + xa;
#pragma unroll
    for (int q = 0; q < (ROWS * WORDS + 31) / 32; ++q) {
      const int i = lane + 32 * q;
      const int r = WORDS == 9 ? (i * 57) >> 9 : (i * 147) >> 10;      // i / WORDS for i < 288 (9) / 192 (7)
      const int k = i - r * WORDS;
      if (r < ROWS && k < nw)
        asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(sa + r * SPITCH + 4 * k), "l"(src + (int64_t)r * pitch + 4 * k) : "memory");
    }
    return x0 & 3;
  }
  stage_footprint_bytes(smem, img, cols, rows, pitch, x0, y0, lane, W, ROWS, SPITCH);
  return 0;
}
__device__ __forceinline__ void stage_wait() {
  asm volatile("cp.async.wait_all;" ::: "memory");
  __syncwarp();
}

// Region-of-interest pyramids (agt_build_pyramid_roi): a pixel of level l >= 1 is exact iff the level-0 support of its
// pyrDown chain, 2^l x +- (2^(l+1) - 2), lies inside the frame's level-0 rectangle (or is cut by the image border, where
// the chain reflects back inside).  Level 0 is the frame itself.  -> half-open window [lo, hi) of exact pixels along one axis.
__device__ __forceinline__ void exact_window(int r_lo, int r_hi, int n0, int n, int level, int& lo, int& hi) {
  if (level == 0) { lo = 0; hi = n; return; }
  const int reach = (2 << level) - 2;
  lo = r_lo <= 0 ? 0 : (r_lo + reach + (1 << level) - 1) >> level;
  hi = r_hi >= n0 ? n : ((r_hi - 1 - reach) >> level) + 1;
  if (hi < 0) hi = 0;
}
// does the footprint [f0, f1) of an n-pixel axis, read with BORDER_REFLECT_101, stay inside [lo, hi)?
__device__ __forceinline__ bool footprint_inside(int f0, int f1, int n, int lo, int hi) {
  int a = max(f0, 0), b = min(f1, n);
  if (f0 < 0) b = max(b, min(n, 1 - f0));                 // -k reads k
  if (f1 > n) a = min(a, max(0, 2 * n - 1 - f1));         // n-1+k reads n-1-k
  return a >= lo && b <= hi;
}

// rects_prev / rects_next (may be null: every level is complete) are the level-0 rectangles the two pyramids were built
// under; a corner whose footprints leave the exact part of a level is flagged in left_roi_out (its outputs are then
// meaningless and the caller redoes the frame on complete pyramids).  mask (may be null): only frames with a non-zero
// entry are processed, the outputs of the others are left untouched.
// Scharr of a window that is cut by the image border: zero outside the image (rare, kept out of line like the byte-wise staging)
__device__ __noinline__ void scharr_cut_window(WarpSmem& S, int ix, int iy, int cols, int rows, int pxo, int lane) {
  for (int i = lane; i < DER * DER; i += 32) {
    int r = i / DER, c = i - r * DER;
    int gx = ix + c, gy = iy + r;
    short2 d = make_short2(0, 0);
    if (gx >= 0 && gx < cols && gy >= 0 && gy < rows) {
      const uint8_t* p = S.u.t.patch + r * PATCH_PITCH + pxo + c;
      int a00 = p[0], a01 = p[1], a02 = p[2];
      int a10 = p[PATCH_PITCH], a12 = p[PATCH_PITCH + 2];
      int a20 = p[2 * PATCH_PITCH], a21 = p[2 * PATCH_PITCH + 1], a22 = p[2 * PATCH_PITCH + 2];
      d.x = (short)(3 * (a02 - a00) + 10 * (a12 - a10) + 3 * (a22 - a20));
      d.y = (short)(3 * (a20 - a00) + 10 * (a21 - a01) + 3 * (a22 - a02));
    }
    S.u.t.der[r][c] = d;
  }
}

// kSplit (lk_levels_kernel, small batches): one warp per pyramid LEVEL of the corner.  What a level prepares - template
// footprint, Scharr window, bilinear template, structure tensor - depends on the corner alone, not on the flow, and is half
// of a corner's instructions: the warps of a CTA prepare all levels at once, then the search runs level by level, each warp
// taking the flow of the level above over from shared memory (handover / publish: a chain of CTA barriers).  The arithmetic
// of every level is the code below either way, so the results are bit-identical.
template <bool kRoi, bool kSplit = false>
__device__ __forceinline__ void lk_corner(WarpSmem& S, const int lane, const int64_t gid, const agt_pyramid& prev, const agt_pyramid& next,
                                          const float* __restrict__ prev_pts, float* __restrict__ next_pts,
                                          uint8_t* __restrict__ status_out, float* __restrict__ err_out, int n_pts,
                                          const int32_t* __restrict__ skip_if_tags_ge2, const int32_t* __restrict__ rects_prev,
                                          const int32_t* __restrict__ rects_next, int rect_stride, const uint8_t* __restrict__ mask,
                                          uint8_t* __restrict__ left_roi_out, const int my_level = 0, float* s_flow = nullptr) {
  static_assert(!(kRoi && kSplit), "the level-parallel variant is for complete pyramids");
  const int frame = (int)(gid / n_pts);
  if (mask != nullptr && mask[frame] == 0) return;
  // region-of-interest rectangles: element k of the previous / next pyramid's rectangle lives in lane k / 4 + k (one
  // register, one exposed load latency per corner) and is fetched by shuffle at every level
  int rect_elem = (lane & 3) < 2 ? 0 : ((lane & 3) == 2 ? prev.width[0] : prev.height[0]);
  if (kRoi) {
    if (lane == 0) S.left = 0;
    if (lane < 4 && rects_prev != nullptr) rect_elem = __ldg(rects_prev + (int64_t)frame * rect_stride + lane);
    if (lane >= 4 && lane < 8 && rects_next != nullptr) rect_elem = __ldg(rects_next + (int64_t)frame * rect_stride + lane - 4);
  }
  if (skip_if_tags_ge2 != nullptr && skip_if_tags_ge2[frame] >= 2) {     // stage-2 rule: tracking only backs up frames with < 2 tags
    if (lane == 0) {
      next_pts[gid * 2] = prev_pts[gid * 2]; next_pts[gid * 2 + 1] = prev_pts[gid * 2 + 1]; status_out[gid] = 0; err_out[gid] = 0.f;
      if (left_roi_out != nullptr) left_roi_out[gid] = 0;
    }
    return;
  }
  const float ptx = prev_pts[gid * 2], pty = prev_pts[gid * 2 + 1];

  float outx = 0.f, outy = 0.f;
  int status = 1;
  float err = 0.f;
  const int top = prev.levels - 1;
  // level-parallel variant: barrier k (k = 1 .. top + 1) lies between the search of level top + 1 - k and that of the level below
  auto cta_barrier = [] { asm volatile("bar.sync 1;" ::: "memory"); };
  auto handover = [&](int level, float px0, float py0, float& nx, float& ny) {
    if (!kSplit) return;
    for (int l = top; l > level; --l) cta_barrier();
    if (level == top) { nx = px0; ny = py0; } else { nx = __fmul_rn(s_flow[0], 2.f); ny = __fmul_rn(s_flow[1], 2.f); }
    outx = nx; outy = ny;
  };
  auto publish = [&](int level) {
    if (!kSplit) return;
    if (lane == 0) { s_flow[0] = outx; s_flow[1] = outy; }
    for (int l = level; l >= 0; --l) cta_barrier();
  };

  for (int level = kSplit ? my_level : top; level >= (kSplit ? my_level : 0); --level) {
    const int cols = prev.width[level], rows = prev.height[level];
    const uint8_t* imgI = prev.data[level] + (int64_t)frame * prev.frame_stride[level];
    const uint8_t* imgJ = next.data[level] + (int64_t)frame * next.frame_stride[level];
    const int64_t pitchI = prev.pitch[level], pitchJ = next.pitch[level];
    const float sc = (float)(1.0 / (double)(1 << level));
    float px = __fmul_rn(ptx, sc), py = __fmul_rn(pty, sc);
    const float px0 = px, py0 = py;
    float nx = 0.f, ny = 0.f;
    if (!kSplit) {
      if (level == top) { nx = px; ny = py; } else { nx = __fmul_rn(outx, 2.f); ny = __fmul_rn(outy, 2.f); }
      outx = nx; outy = ny;
    }
    px = __fsub_rn(px, 10.f); py = __fsub_rn(py, 10.f);
    const int ix = (int)floorf(px), iy = (int)floorf(py);
    // also rejects NaN / huge coordinates (the float->int conversion saturates)
    if (!(px == px) || !(py == py) || ix < -WIN || ix >= cols || iy < -WIN || iy >= rows) {
      if (level == 0) { status = 0; err = 0.f; }
      handover(level, px0, py0, nx, ny);
      publish(level);
      continue;
    }
    if (kRoi) {
      int rp[4], rn[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) { rp[k] = __shfl_sync(0xffffffffu, rect_elem, k); rn[k] = __shfl_sync(0xffffffffu, rect_elem, 4 + k); }
      int ax, bx, ay, by;
      exact_window(rp[0], rp[2], prev.width[0], cols, level, ax, bx);
      exact_window(rp[1], rp[3], prev.height[0], rows, level, ay, by);
      const bool out = !footprint_inside(ix - 1, ix - 1 + PATCH, cols, ax, bx) || !footprint_inside(iy - 1, iy - 1 + PATCH, rows, ay, by);
      exact_window(rn[0], rn[2], prev.width[0], cols, level, ax, bx);
      exact_window(rn[1], rn[3], prev.height[0], rows, level, ay, by);
      __syncwarp();
      if (lane == 0) { S.win[0] = ax; S.win[1] = bx; S.win[2] = ay; S.win[3] = by; if (out) S.left = 1; }
    }
    __syncwarp();
    // ---- stage the 24x24 template footprint (reflect-101 intensity) -------------
    // (requesting the next level's footprint during this level's search - its position depends only on the corner - was
    // measured slower, 1.25 against 1.15 ms per 98k corners: one more live register under the 64-register cap)
    const int pxo = stage_footprint<PATCH, PATCH, 7, PATCH_PITCH>(S.u.t.patch, imgI, cols, rows, pitchI, ix - 1, iy - 1, lane);
    stage_wait();
    // ---- Scharr at the 22x22 integer positions; zero outside the image -------------
    if (ix >= 0 && iy >= 0 && ix + DER <= cols && iy + DER <= rows) {
      // window inside the image (warp-uniform): a lane per row reads the three footprint rows as aligned words and
      // forms every derivative with chained dp4a ([3 10 3] folded into the byte coefficients), no per-tap byte loads
      if (lane < DER) {
        uint32_t w[3][PATCH / 4];
        const uint32_t psh = (uint32_t)pxo * 8u;
#pragma unroll
        for (int rr = 0; rr < 3; ++rr) {
          const uint32_t* src = reinterpret_cast<const uint32_t*>(&S.u.t.patch[(lane + rr) * PATCH_PITCH]);      // 7 aligned words
          uint32_t t[PATCH / 4 + 1];
#pragma unroll
          for (int q = 0; q <= PATCH / 4; ++q) t[q] = src[q];
#pragma unroll
          for (int q = 0; q < PATCH / 4; ++q) w[rr][q] = __funnelshift_r(t[q], t[q + 1], psh);
        }
#pragma unroll
        for (int c = 0; c < DER; ++c) {
          const int j = c >> 2, m = c & 3;              // bytes c..c+2 of a row = bytes m..m+2 of word j (and word j+1)
          // coefficient words for a tap triple starting at byte m: difference (-k, 0, +k) and smoothing (3, 10, 3)
          const int d3a = m == 0 ? 0x000300FD : m == 1 ? 0x0300FD00 : m == 2 ? (int)0x00FD0000 : (int)0xFD000000;
          const int d3b = m == 2 ? 0x00000003 : m == 3 ? 0x00000300 : 0;
          const int d10a = m == 0 ? 0x000A00F6 : m == 1 ? 0x0A00F600 : m == 2 ? (int)0x00F60000 : (int)0xF6000000;
          const int d10b = m == 2 ? 0x0000000A : m == 3 ? 0x00000A00 : 0;
          const int sma = m == 0 ? 0x00030A03 : m == 1 ? 0x030A0300 : m == 2 ? 0x0A030000 : 0x03000000;
          const int smb = m == 2 ? 0x00000003 : m == 3 ? 0x0000030A : 0;
          const int nsma = m == 0 ? 0x00FDF6FD : m == 1 ? (int)0xFDF6FD00 : m == 2 ? (int)0xF6FD0000 : (int)0xFD000000;
          const int nsmb = m == 2 ? 0x000000FD : m == 3 ? 0x0000FDF6 : 0;
          int dx = dp4us(w[2][j], d3a, dp4us(w[1][j], d10a, dp4us(w[0][j], d3a, 0)));
          int dy = dp4us(w[2][j], sma, dp4us(w[0][j], nsma, 0));
          if (m >= 2) {
            dx = dp4us(w[2][j + 1], d3b, dp4us(w[1][j + 1], d10b, dp4us(w[0][j + 1], d3b, dx)));
            dy = dp4us(w[2][j + 1], smb, dp4us(w[0][j + 1], nsmb, dy));
          }
          S.u.t.der[lane][c] = make_short2((short)dx, (short)dy);
        }
      }
    } else {
      scharr_cut_window(S, ix, iy, cols, rows, pxo, lane);
    }
    __syncwarp();
    // ---- template + structure tensor (lane-major pixel order, see WarpSmem) ------------------
    Weights w = make_weights(__fsub_rn(px, (float)ix), __fsub_rn(py, (float)iy));
    const bool row_lane = lane < WIN;
    int seg_row[2], seg_col[2];
    segment_of(lane, 0, seg_row[0], seg_col[0]);
    segment_of(lane, 1, seg_row[1], seg_col[1]);
    const uint32_t patch_a = (uint32_t)__cvta_generic_to_shared(&S.u.t.patch[0]) + pxo;
    const uint32_t wtI = ((uint32_t)w.w00 & 0xffffu) | ((uint32_t)w.w01 << 16), wbI = ((uint32_t)w.w10 & 0xffffu) | ((uint32_t)w.w11 << 16);
    int4* const ddl = &S.dd[lane];
#pragma unroll
    for (int sg = 0; sg < 2; ++sg) {
      const bool live = seg_row[sg] < WIN;
      const int y = live ? seg_row[sg] : WIN - 1, x0 = seg_col[sg];
      // the run's template intensities: rows y+1, y+2 of the footprint from column x0+1, blended as in the search loop
      const Run t = load_run(patch_a + (y + 1) * PATCH_PITCH + x0 + 1), bt = load_run(patch_a + (y + 2) * PATCH_PITCH + x0 + 1);
      int ivs[SEG_LEN];
      ivs[0] = blend<0>(t, bt, wtI, wbI); ivs[1] = blend<1>(t, bt, wtI, wbI); ivs[2] = blend<2>(t, bt, wtI, wbI);
      ivs[3] = blend<3>(t, bt, wtI, wbI); ivs[4] = blend<4>(t, bt, wtI, wbI); ivs[5] = blend<5>(t, bt, wtI, wbI);
      ivs[6] = blend<6>(t, bt, wtI, wbI); ivs[7] = blend<7>(t, bt, wtI, wbI);
      // the Scharr values of the run's two rows, each used by two neighbouring pixels (a tail lane needs six per row)
      short2 d0[SEG_LEN + 1], d1[SEG_LEN + 1];
#pragma unroll
      for (int k = 0; k <= SEG_LEN; ++k) {
        const int c = row_lane || k <= TAIL_LEN ? x0 + k : x0;
        d0[k] = S.u.t.der[y][c]; d1[k] = S.u.t.der[y + 1][c];
      }
      int dxs[SEG_LEN], dys[SEG_LEN];
#pragma unroll
      for (int k = 0; k < SEG_LEN; ++k) {
        dxs[k] = descale(d0[k].x * w.w00 + d0[k + 1].x * w.w01 + d1[k].x * w.w10 + d1[k + 1].x * w.w11, W_BITS);
        dys[k] = descale(d0[k].y * w.w00 + d0[k + 1].y * w.w01 + d1[k].y * w.w10 + d1[k + 1].y * w.w11, W_BITS);
        if (!live || !(row_lane || k < TAIL_LEN)) { ivs[k] = 0; dxs[k] = 0; dys[k] = 0; }
      }
      S.tmpl[sg][lane] = make_uint4((uint32_t)(ivs[0] & 0xffff) | ((uint32_t)ivs[1] << 16), (uint32_t)(ivs[2] & 0xffff) | ((uint32_t)ivs[3] << 16),
                                    (uint32_t)(ivs[4] & 0xffff) | ((uint32_t)ivs[5] << 16), (uint32_t)(ivs[6] & 0xffff) | ((uint32_t)ivs[7] << 16));
#pragma unroll
      for (int pr = 0; pr < 4; ++pr)
        if (pr < 3 || row_lane) ddl[sg * DD_RUN + (pr < 3 ? 32 * pr : 96)] = make_int4(dxs[2 * pr], dys[2 * pr], dxs[2 * pr + 1], dys[2 * pr + 1]);
    }
    __syncwarp();      // der / patch are dead from here on: the float scratch of the ordered sums overlays them
    // ---- structure tensor, summed in float32 in OpenCV's order (see the header) -------------------------------------------
    // (dx, dy) of column c (0..15) of this row lane / of tail pixel i (0..9) of this tail lane
#define AGT_DD_COL(c) (reinterpret_cast<const int2*>(&ddl[((c) >> 3) * DD_RUN + ((((c) & 7) >> 1) < 3 ? 32 * (((c) & 7) >> 1) : 96)])[(c) & 1])
#define AGT_DD_TAIL(i) (reinterpret_cast<const int2*>(&ddl[((i) / TAIL_LEN) * DD_RUN + 32 * (((i) % TAIL_LEN) >> 1)])[((i) % TAIL_LEN) & 1])
    // pass 1: A11 and A12 of columns 0..15 (lanes 0..3 / 4..7 run the SIMD lane chains: 84 additions each)
    if (row_lane) {
#pragma unroll
      for (int kk = 0; kk < 4; ++kk) {
        float fx[4], fy[4];
#pragma unroll
        for (int m = 0; m < 4; ++m) { const int2 d = AGT_DD_COL(4 * m + kk); fx[m] = (float)d.x; fy[m] = (float)d.y; }
        // |d| <= 4080: the products are below 2^24, i.e. exact
        *reinterpret_cast<float4*>(&S.u.a1.simd[kk][4 * lane]) = make_float4(fx[0] * fx[0], fx[1] * fx[1], fx[2] * fx[2], fx[3] * fx[3]);
        *reinterpret_cast<float4*>(&S.u.a1.simd[4 + kk][4 * lane]) = make_float4(fx[0] * fy[0], fx[1] * fy[1], fx[2] * fy[2], fx[3] * fy[3]);
      }
    }
    __syncwarp();
    float acc = 0.f;
    if (lane < 8) acc = ordered_sum<CH_A / 4>(reinterpret_cast<const float4*>(S.u.a1.simd[lane]), 0.f);
    acc = reduce_lanes4(acc);
    const float A11s = __shfl_sync(0xffffffffu, acc, 0), A12s = __shfl_sync(0xffffffffu, acc, 4);
    __syncwarp();
    // pass 2: A22 of columns 0..15 (lanes 0..3) and the scalar tails of A11, A12, A22 (lanes 4..6: 105 additions each)
    if (row_lane) {
#pragma unroll
      for (int kk = 0; kk < 4; ++kk) {
        float fy[4];
#pragma unroll
        for (int m = 0; m < 4; ++m) fy[m] = (float)AGT_DD_COL(4 * m + kk).y;
        *reinterpret_cast<float4*>(&S.u.a2.simd[kk][4 * lane]) = make_float4(fy[0] * fy[0], fy[1] * fy[1], fy[2] * fy[2], fy[3] * fy[3]);
      }
    } else {
      // ten tail pixels: rows 2j, 2j+1 -> elements 10 j .. 10 j + 9 of each tail chain (lane 31's second row is zero: the
      // zero padding of the chains; CH_ATAIL leaves room for it)
      float f11[2 * TAIL_LEN], f12[2 * TAIL_LEN], f22[2 * TAIL_LEN];
#pragma unroll
      for (int i = 0; i < 2 * TAIL_LEN; ++i) {
        const int2 d = AGT_DD_TAIL(i);
        const float fx = (float)d.x, fy = (float)d.y;
        f11[i] = fx * fx; f12[i] = fx * fy; f22[i] = fy * fy;
      }
      const int e = 2 * TAIL_LEN * (lane - WIN);
#pragma unroll
      for (int i = 0; i < TAIL_LEN; ++i) {
        *reinterpret_cast<float2*>(&S.u.a2.tail[0][e + 2 * i]) = make_float2(f11[2 * i], f11[2 * i + 1]);
        *reinterpret_cast<float2*>(&S.u.a2.tail[1][e + 2 * i]) = make_float2(f12[2 * i], f12[2 * i + 1]);
        *reinterpret_cast<float2*>(&S.u.a2.tail[2][e + 2 * i]) = make_float2(f22[2 * i], f22[2 * i + 1]);
      }
    }
#undef AGT_DD_COL
#undef AGT_DD_TAIL
    __syncwarp();
    acc = 0.f;
    if (lane < 4) acc = ordered_sum<CH_A / 4>(reinterpret_cast<const float4*>(S.u.a2.simd[lane]), 0.f);
    else if (lane < 7) acc = ordered_sum<CH_TAIL / 4>(reinterpret_cast<const float4*>(S.u.a2.tail[lane - 4]), 0.f);
    const float A22s = __shfl_sync(0xffffffffu, reduce_lanes4(acc), 0);
    const float FLT_SCALE = 1.f / (float)(1 << 20);
    float A11 = __fmul_rn(__fadd_rn(__shfl_sync(0xffffffffu, acc, 4), A11s), FLT_SCALE);
    float A12 = __fmul_rn(__fadd_rn(__shfl_sync(0xffffffffu, acc, 5), A12s), FLT_SCALE);
    float A22 = __fmul_rn(__fadd_rn(__shfl_sync(0xffffffffu, acc, 6), A22s), FLT_SCALE);
    float D = __fsub_rn(__fmul_rn(A11, A22), __fmul_rn(A12, A12));
    float dif = __fsub_rn(A11, A22);
    float disc = __fadd_rn(__fmul_rn(dif, dif), __fmul_rn(__fmul_rn(4.f, A12), A12));
    float minEig = __fdiv_rn(__fsub_rn(__fadd_rn(A22, A11), __fsqrt_rn(disc)), (float)(2 * WIN * WIN));
    if ((double)minEig < 1e-4 || D < 1.1920928955078125e-7f) {
      if (level == 0) status = 0;
      handover(level, px0, py0, nx, ny);
      publish(level);
      continue;
    }
    D = __fdiv_rn(1.f, D);
    handover(level, px0, py0, nx, ny);       // (level-parallel variant: wait for the flow of the level above)
    __syncwarp();      // the scratch of the tensor sums is dead: the region buffer and the search scratch may overwrite it
    // zero padding of the search chains (elements 42, 43 of the eight lane chains; the tail's comes from lane 31's dead row)
    if (lane < 8) *reinterpret_cast<float2*>(&S.u.region.simd[lane][CH_SIMD - 2]) = make_float2(0.f, 0.f);

    const uint32_t region_a = (uint32_t)__cvta_generic_to_shared(&S.u.region.px[0]);
    int rxo = 0;                               // byte offset of column rx0 inside a staged row
    // shared-memory offset of each run inside the region for a window at (0, 0); disabled runs read a valid row
    const int run_off0 = (seg_row[0] < WIN ? seg_row[0] : WIN - 1) * REG_PITCH + seg_col[0];
    const int run_off1 = (seg_row[1] < WIN ? seg_row[1] : WIN - 1) * REG_PITCH + seg_col[1];
    const float4* chain = lane < 8 ? reinterpret_cast<const float4*>(S.u.region.simd[lane])
                                   : reinterpret_cast<const float4*>(S.u.region.tail[lane & 1]);

    nx = __fsub_rn(nx, 10.f); ny = __fsub_rn(ny, 10.f);
    float pdx = 0.f, pdy = 0.f;
    int rx0 = 0, ry0 = 0;
    bool staged = false;
    for (int j = 0; j < MAX_ITERS; ++j) {
      int jx = (int)floorf(nx), jy = (int)floorf(ny);
      if (!(nx == nx) || !(ny == ny) || jx < -WIN || jx >= cols || jy < -WIN || jy >= rows) {
        if (level == 0) status = 0;
        break;
      }
      if (!staged || jx < rx0 || jx > rx0 + (REG - DER) || jy < ry0 || jy > ry0 + (REG_H - DER)) {
        __syncwarp();
        rx0 = jx - REG_MARGIN; ry0 = jy - REG_MARGIN_Y;
        if (kRoi) {
          const int4 wn = *reinterpret_cast<const int4*>(S.win);
          if (lane == 0 && (!footprint_inside(rx0, rx0 + REG, cols, wn.x, wn.y) || !footprint_inside(ry0, ry0 + REG_H, rows, wn.z, wn.w))) S.left = 1;
        }
        rxo = stage_footprint<REG, REG_H, 9, REG_PITCH>(S.u.region.px, imgJ, cols, rows, pitchJ, rx0, ry0, lane);
        staged = true;
        stage_wait();
      }
      Weights wj = make_weights(__fsub_rn(nx, (float)jx), __fsub_rn(ny, (float)jy));
      const uint32_t wt = ((uint32_t)wj.w00 & 0xffffu) | ((uint32_t)wj.w01 << 16), wb = ((uint32_t)wj.w10 & 0xffffu) | ((uint32_t)wj.w11 << 16);
      const uint32_t win_a = region_a + (jy - ry0) * REG_PITCH + (jx - rx0) + rxo;
      // mismatch products (J - I) dI per pixel: exact integers; pf holds what goes into the float chains - a row lane's
      // four pair sums (columns k, k+4) per run and component, a tail lane's five single products per run and component
      // (the two runs of a lane as a rolled loop - half the code of the iteration, 32-bit stores - measured 2 % slower: 8.43 / 8.28 ms)
      float pfx[2][TAIL_LEN], pfy[2][TAIL_LEN];
#pragma unroll
      for (int sg = 0; sg < 2; ++sg) {
        const uint32_t a = win_a + (sg == 0 ? run_off0 : run_off1);
        const Run t = load_run(a), bt = load_run(a + REG_PITCH);
        int jv[SEG_LEN];
        jv[0] = blend<0>(t, bt, wt, wb); jv[1] = blend<1>(t, bt, wt, wb); jv[2] = blend<2>(t, bt, wt, wb);
        jv[3] = blend<3>(t, bt, wt, wb); jv[4] = blend<4>(t, bt, wt, wb); jv[5] = blend<5>(t, bt, wt, wb);
        jv[6] = blend<6>(t, bt, wt, wb); jv[7] = blend<7>(t, bt, wt, wb);
        const uint4 tq = S.tmpl[sg][lane];
        const uint32_t tw[4] = {tq.x, tq.y, tq.z, tq.w};
        int sx[SEG_LEN], sy[SEG_LEN];
#pragma unroll
        for (int k = 0; k < SEG_LEN; ++k) {
          const int4 d2 = ddl[sg * DD_RUN + ((k >> 1) < 3 ? 32 * (k >> 1) : 96)];
          const int dx = (k & 1) ? d2.z : d2.x, dy = (k & 1) ? d2.w : d2.y;
          const int ti = (k & 1) ? (int)tw[k >> 1] >> 16 : (int)(short)(tw[k >> 1] & 0xffffu);
          const int diff = jv[k] - ti;
          sx[k] = diff * dx; sy[k] = diff * dy;         // |diff| <= 8160, |d| <= 4080
        }
        if (row_lane) {
#pragma unroll
          for (int k = 0; k < 4; ++k) { pfx[sg][k] = (float)(sx[k] + sx[k + 4]); pfy[sg][k] = (float)(sy[k] + sy[k + 4]); }   // pmaddwd + cvtdq2ps
        } else {
#pragma unroll
          for (int k = 0; k < TAIL_LEN; ++k) { pfx[sg][k] = (float)sx[k]; pfy[sg][k] = (float)sy[k]; }
        }
      }
      if (row_lane) {
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          *reinterpret_cast<float2*>(&S.u.region.simd[k][2 * lane]) = make_float2(pfx[0][k], pfx[1][k]);
          *reinterpret_cast<float2*>(&S.u.region.simd[4 + k][2 * lane]) = make_float2(pfy[0][k], pfy[1][k]);
        }
      } else {
        const int e = 2 * TAIL_LEN * (lane - WIN);
        const float ox[2 * TAIL_LEN] = {pfx[0][0], pfx[0][1], pfx[0][2], pfx[0][3], pfx[0][4], pfx[1][0], pfx[1][1], pfx[1][2], pfx[1][3], pfx[1][4]};
        const float oy[2 * TAIL_LEN] = {pfy[0][0], pfy[0][1], pfy[0][2], pfy[0][3], pfy[0][4], pfy[1][0], pfy[1][1], pfy[1][2], pfy[1][3], pfy[1][4]};
#pragma unroll
        for (int i = 0; i < TAIL_LEN; ++i) {
          if (e + 2 * i < CH_TAIL) {           // lane 31's dead row supplies the zeros 105..107; 108, 109 do not exist
            *reinterpret_cast<float2*>(&S.u.region.tail[0][e + 2 * i]) = make_float2(ox[2 * i], ox[2 * i + 1]);
            *reinterpret_cast<float2*>(&S.u.region.tail[1][e + 2 * i]) = make_float2(oy[2 * i], oy[2 * i + 1]);
          }
        }
      }
      __syncwarp();
      // the ten dependent chains: lanes 0..3 x / 4..7 y of the SIMD lanes (42 additions), lanes 8, 9 the scalar tails (105)
      float ch = 0.f;
      if (lane < 10) {
        ch = ordered_sum<CH_SIMD / 4>(chain, 0.f);
        if (lane >= 8) ch = ordered_sum<(CH_TAIL - CH_SIMD) / 4>(chain + CH_SIMD / 4, ch);
      }
      const float lanes4 = reduce_lanes4(ch);
      const float ib1 = __fadd_rn(__shfl_sync(0xffffffffu, ch, 8), __shfl_sync(0xffffffffu, lanes4, 0));
      const float ib2 = __fadd_rn(__shfl_sync(0xffffffffu, ch, 9), __shfl_sync(0xffffffffu, lanes4, 4));
      __syncwarp();
      float b1 = __fmul_rn(ib1, FLT_SCALE);
      float b2 = __fmul_rn(ib2, FLT_SCALE);
      float dx = __fmul_rn(__fsub_rn(__fmul_rn(A12, b2), __fmul_rn(A22, b1)), D);
      float dy = __fmul_rn(__fsub_rn(__fmul_rn(A12, b1), __fmul_rn(A11, b2)), D);
      nx = __fadd_rn(nx, dx); ny = __fadd_rn(ny, dy);
      outx = __fadd_rn(nx, 10.f); outy = __fadd_rn(ny, 10.f);
      if ((double)dx * (double)dx + (double)dy * (double)dy <= 0.01 * 0.01) break;
      if (j > 0 && fabs((double)__fadd_rn(dx, pdx)) < 0.01 && fabs((double)__fadd_rn(dy, pdy)) < 0.01) {
        outx = __fsub_rn(outx, __fmul_rn(dx, 0.5f));
        outy = __fsub_rn(outy, __fmul_rn(dy, 0.5f));
        break;
      }
      pdx = dx; pdy = dy;
    }

    if (status && level == 0) {
      float ex = __fsub_rn(outx, 10.f), ey = __fsub_rn(outy, 10.f);
      int jx = (int)floorf(ex), jy = (int)floorf(ey);
      if (!(ex == ex) || !(ey == ey) || jx < -WIN || jx >= cols || jy < -WIN || jy >= rows) {
        status = 0;
      } else {
        if (!staged || jx < rx0 || jx > rx0 + (REG - DER) || jy < ry0 || jy > ry0 + (REG_H - DER)) {
          __syncwarp();
          rx0 = jx - REG_MARGIN; ry0 = jy - REG_MARGIN_Y;
          if (kRoi) {
            const int4 wn = *reinterpret_cast<const int4*>(S.win);
            if (lane == 0 && (!footprint_inside(rx0, rx0 + REG, cols, wn.x, wn.y) || !footprint_inside(ry0, ry0 + REG_H, rows, wn.z, wn.w))) S.left = 1;
          }
          rxo = stage_footprint<REG, REG_H, 9, REG_PITCH>(S.u.region.px, imgJ, cols, rows, pitchJ, rx0, ry0, lane);
          stage_wait();
        }
        Weights wj = make_weights(__fsub_rn(ex, (float)jx), __fsub_rn(ey, (float)jy));
        const uint32_t wt = ((uint32_t)wj.w00 & 0xffffu) | ((uint32_t)wj.w01 << 16), wb = ((uint32_t)wj.w10 & 0xffffu) | ((uint32_t)wj.w11 << 16);
        const uint32_t win_a = region_a + (jy - ry0) * REG_PITCH + (jx - rx0) + rxo;
        int sabs = 0;          // sum of |diff| <= 441 * 8160 < 2^24: exact in OpenCV's float accumulator whatever the order
#pragma unroll
        for (int sg = 0; sg < 2; ++sg) {
          if (seg_row[sg] >= WIN) continue;
          const uint32_t a = win_a + (sg == 0 ? run_off0 : run_off1);
          const Run t = load_run(a), bt = load_run(a + REG_PITCH);
          int jv[SEG_LEN];
          jv[0] = blend<0>(t, bt, wt, wb); jv[1] = blend<1>(t, bt, wt, wb); jv[2] = blend<2>(t, bt, wt, wb);
          jv[3] = blend<3>(t, bt, wt, wb); jv[4] = blend<4>(t, bt, wt, wb); jv[5] = blend<5>(t, bt, wt, wb);
          jv[6] = blend<6>(t, bt, wt, wb); jv[7] = blend<7>(t, bt, wt, wb);
          const uint4 tq = S.tmpl[sg][lane];
          const uint32_t tw[4] = {tq.x, tq.y, tq.z, tq.w};
#pragma unroll
          for (int k = 0; k < SEG_LEN; ++k) {
            const int diff = jv[k] - ((k & 1) ? (int)tw[k >> 1] >> 16 : (int)(short)(tw[k >> 1] & 0xffffu));
            if (row_lane || k < TAIL_LEN) sabs += diff < 0 ? -diff : diff;
          }
        }
        err = __fdiv_rn((float)warp_sum_wide(sabs), (float)(32 * WIN * WIN));      // `errval * 1.f / (32 * w * h)`
      }
    }
    publish(level);
  }
  if (lane == 0 && (!kSplit || my_level == 0)) {
    next_pts[gid * 2] = outx;
    next_pts[gid * 2 + 1] = outy;
    status_out[gid] = (uint8_t)status;
    err_out[gid] = status ? err : 0.f;
    if (kRoi && left_roi_out != nullptr) left_roi_out[gid] = S.left ? 1 : 0;
  }
}

// One warp per corner.  Unmasked launches have one corner per warp; masked launches (the redo pass of agt_lk_roi: few
// frames flagged, usually none) use a small grid whose warps stride over the corners and leave after one pass over the
// mask when nothing is flagged, instead of launching tens of thousands of CTAs that have nothing to do.
template <bool kRoi, bool kStride>
__global__ void __launch_bounds__(WARPS_PER_CTA * 32, 4)
lk_kernel(agt_pyramid prev, agt_pyramid next, const float* __restrict__ prev_pts, float* __restrict__ next_pts,
          uint8_t* __restrict__ status_out, float* __restrict__ err_out, int n_pts, int64_t total,
          const int32_t* __restrict__ skip_if_tags_ge2, const int32_t* __restrict__ rects_prev,
          const int32_t* __restrict__ rects_next, int rect_stride, const uint8_t* __restrict__ mask,
          uint8_t* __restrict__ left_roi_out) {
  extern __shared__ __align__(16) uint8_t lk_smem_raw[];      // WARPS_PER_CTA x WarpSmem (more than the 48 KB static limit)
  WarpSmem* smem = reinterpret_cast<WarpSmem*>(lk_smem_raw);
  const int lane = threadIdx.x & 31;
  const int wid = threadIdx.x >> 5;
  if (!kStride) {
    const int64_t gid = (int64_t)blockIdx.x * WARPS_PER_CTA + wid;
    if (gid < total)
      lk_corner<kRoi>(smem[wid], lane, gid, prev, next, prev_pts, next_pts, status_out, err_out, n_pts, skip_if_tags_ge2, rects_prev,
                      rects_next, rect_stride, mask, left_roi_out);
    return;
  }
  if (mask != nullptr) {
    const int64_t n_frames = total / n_pts;
    uint32_t acc = 0;
    for (int64_t i = threadIdx.x; i < n_frames; i += blockDim.x) acc |= mask[i];
    if (!__syncthreads_or(acc != 0)) return;
  }
  for (int64_t gid = (int64_t)blockIdx.x * WARPS_PER_CTA + wid; gid < total; gid += (int64_t)gridDim.x * WARPS_PER_CTA) {
    lk_corner<kRoi>(smem[wid], lane, gid, prev, next, prev_pts, next_pts, status_out, err_out, n_pts, skip_if_tags_ge2, rects_prev,
                    rects_next, rect_stride, mask, left_roi_out);
    __syncwarp();
  }
}

// Small batches (the stream pipeline tracks a few hundred corners per step, and waits for them): a CTA per corner, a warp per
// pyramid level - see lk_corner<kRoi, kSplit>.  Same outputs as lk_kernel bit for bit, about half its latency.
__global__ void __launch_bounds__(AGT_MAX_LEVELS * 32)
lk_levels_kernel(agt_pyramid prev, agt_pyramid next, const float* __restrict__ prev_pts, float* __restrict__ next_pts,
                 uint8_t* __restrict__ status_out, float* __restrict__ err_out, int n_pts, const int32_t* __restrict__ skip_if_tags_ge2) {
  extern __shared__ __align__(16) uint8_t lk_smem_raw[];      // one WarpSmem per level
  __shared__ float s_flow[2];
  WarpSmem* smem = reinterpret_cast<WarpSmem*>(lk_smem_raw);
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  lk_corner<false, true>(smem[wid], lane, (int64_t)blockIdx.x, prev, next, prev_pts, next_pts, status_out, err_out, n_pts, skip_if_tags_ge2,
                         nullptr, nullptr, 0, nullptr, nullptr, prev.levels - 1 - wid, s_flow);
}

// Level-0 rectangle (x0,y0,x1,y1; x multiples of 16) that covers what tracking the points of one frame can read when no
// point moves more than max_flow level-0 pixels: per level the 32-pixel search region around the estimate (+-16 level
// pixels, which contains the template footprint), the flow, and the pyrDown chain: (16 + 2) * 2^top + max_flow.
// Points outside the frame are clamped to it (they read the reflected border region at most), NaNs are ignored.
__global__ void lk_rects_kernel(const float* __restrict__ pts, const uint8_t* __restrict__ valid, int n_pts, int W, int H,
                                int top, int max_flow, int32_t* __restrict__ rects, int rect_stride, int batch) {
  const int frame = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (frame >= batch) return;
  int x0 = W, y0 = H, x1 = -1, y1 = -1;
  for (int k = lane; k < n_pts; k += 32) {
    if (valid != nullptr && valid[(int64_t)frame * n_pts + k] == 0) continue;
    const float x = pts[((int64_t)frame * n_pts + k) * 2], y = pts[((int64_t)frame * n_pts + k) * 2 + 1];
    if (!(x == x) || !(y == y)) continue;
    const int xi = (int)fminf(fmaxf(x, 0.f), (float)(W - 1)), yi = (int)fminf(fmaxf(y, 0.f), (float)(H - 1));
    x0 = min(x0, xi); y0 = min(y0, yi); x1 = max(x1, xi); y1 = max(y1, yi);
  }
  for (int o = 16; o > 0; o >>= 1) {
    x0 = min(x0, __shfl_xor_sync(0xffffffffu, x0, o)); y0 = min(y0, __shfl_xor_sync(0xffffffffu, y0, o));
    x1 = max(x1, __shfl_xor_sync(0xffffffffu, x1, o)); y1 = max(y1, __shfl_xor_sync(0xffffffffu, y1, o));
  }
  if (lane == 0) {
    int32_t* r = rects + (int64_t)frame * rect_stride;
    if (x1 < 0) { r[0] = r[1] = r[2] = r[3] = 0; return; }
    const int pad = (18 << top) + max_flow;
    x0 = max(0, x0 - pad) & ~15; y0 = max(0, y0 - pad);
    x1 = min(W, (x1 + 1 + pad + 15) & ~15); y1 = min(H, y1 + 1 + pad);
    r[0] = x0; r[1] = y0; r[2] = x1; r[3] = y1;
  }
}

// Stage-2 integration: one thread per (frame, tag).
__global__ void lk_merge_kernel(const float* __restrict__ tracked, const uint8_t* __restrict__ status,
                                const uint8_t* __restrict__ prev_valid, float* __restrict__ img, uint8_t* __restrict__ valid,
                                int32_t* __restrict__ n_tags, int32_t* __restrict__ tracked_tags, int batch, int tags) {
  int f = blockIdx.x;
  if (f >= batch) return;
  __shared__ int s_cnt;
  if (threadIdx.x == 0) s_cnt = 0;
  __syncthreads();
  const int before = n_tags[f];
  const int need = before < 2;
  int t = threadIdx.x;
  if (t < tags) {
    int64_t base = ((int64_t)f * tags + t) * 4;
    bool det = valid[base] && valid[base + 1] && valid[base + 2] && valid[base + 3];
    if (!det && need) {
      bool ok = true;
      for (int j = 0; j < 4; ++j) ok = ok && prev_valid[base + j] != 0 && status[base + j] == 1;
      if (ok) {
        for (int j = 0; j < 4; ++j) {
          img[(base + j) * 2] = tracked[(base + j) * 2];
          img[(base + j) * 2 + 1] = tracked[(base + j) * 2 + 1];
          valid[base + j] = 1;
        }
        det = true;
      }
    }
    if (det) atomicAdd(&s_cnt, 1);
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    n_tags[f] = s_cnt;
    if (tracked_tags) tracked_tags[f] = s_cnt - before;
  }
}

}  // namespace

extern "C" int agt_lk_merge(agt_ctx* ctx, const float* d_tracked_pts, const uint8_t* d_status, const uint8_t* d_prev_valid,
                            float* d_img_pts, uint8_t* d_valid, int32_t* d_n_tags, int32_t* d_tracked_tags, int batch, int n_pts) {
  if (!ctx) return AGT_ERR_INVALID;
  if (batch == 0) return AGT_OK;          // nothing to do (empty tensors may carry null pointers)
  if (!d_tracked_pts || !d_status || !d_prev_valid || !d_img_pts || !d_valid || !d_n_tags || batch < 0 || n_pts < 4 ||
      (n_pts & 3) || n_pts > AGT_MAX_POINTS)
    AGT_FAIL(ctx, AGT_ERR_INVALID, "agt_lk_merge: bad arguments");
  if (batch == 0) return AGT_OK;
  lk_merge_kernel<<<batch, 32, 0, ctx->stream>>>(d_tracked_pts, d_status, d_prev_valid, d_img_pts, d_valid, d_n_tags, d_tracked_tags, batch,
                                                 n_pts / 4);
  AGT_LAUNCH_CHECK(ctx);
  return AGT_OK;
}

static int lk_impl(agt_ctx* ctx, const agt_pyramid* prev, const agt_pyramid* next, const float* d_prev_pts, float* d_next_pts,
                   uint8_t* d_status, float* d_err, int batch, int n_pts, const int32_t* d_n_tags, const int32_t* d_rects_prev = nullptr,
                   const int32_t* d_rects_next = nullptr, int rect_stride = 0, const uint8_t* d_mask = nullptr,
                   uint8_t* d_left_roi = nullptr);

extern "C" int agt_lk(agt_ctx* ctx, const agt_pyramid* prev, const agt_pyramid* next, const float* d_prev_pts,
                      float* d_next_pts, uint8_t* d_status, float* d_err, int batch, int n_pts) {
  if (!ctx) return AGT_ERR_INVALID;
  return lk_impl(ctx, prev, next, d_prev_pts, d_next_pts, d_status, d_err, batch, n_pts, nullptr);
}

extern "C" int agt_lk_fallback(agt_ctx* ctx, const agt_pyramid* prev, const agt_pyramid* next, const float* d_prev_pts,
                               float* d_next_pts, uint8_t* d_status, float* d_err, const int32_t* d_n_tags, int batch, int n_pts) {
  if (!ctx) return AGT_ERR_INVALID;
  if (!d_n_tags) AGT_FAIL(ctx, AGT_ERR_INVALID, "agt_lk_fallback: d_n_tags is NULL");
  return lk_impl(ctx, prev, next, d_prev_pts, d_next_pts, d_status, d_err, batch, n_pts, d_n_tags);
}

extern "C" int agt_lk_roi(agt_ctx* ctx, const agt_pyramid* prev, const agt_pyramid* next, const float* d_prev_pts,
                          float* d_next_pts, uint8_t* d_status, float* d_err, const int32_t* d_n_tags, const int32_t* d_rects_prev,
                          const int32_t* d_rects_next, int rect_stride, const uint8_t* d_mask, uint8_t* d_left_roi, int batch,
                          int n_pts) {
  if (!ctx) return AGT_ERR_INVALID;
  if ((d_rects_prev || d_rects_next) && rect_stride < 4) AGT_FAIL(ctx, AGT_ERR_INVALID, "agt_lk_roi: rect_stride < 4");
  if ((d_rects_prev || d_rects_next) && !d_left_roi && (int64_t)batch * n_pts > 0)
    AGT_FAIL(ctx, AGT_ERR_INVALID, "agt_lk_roi: d_left_roi is required with region-of-interest pyramids");
  return lk_impl(ctx, prev, next, d_prev_pts, d_next_pts, d_status, d_err, batch, n_pts, d_n_tags, d_rects_prev, d_rects_next,
                 rect_stride, d_mask, d_left_roi);
}

extern "C" int agt_lk_rects(agt_ctx* ctx, const agt_pyramid* pyr, const float* d_pts, const uint8_t* d_valid, int n_pts,
                            int max_flow, int32_t* d_rects, int rect_stride, int batch) {
  if (!ctx) return AGT_ERR_INVALID;
  if (batch == 0) return AGT_OK;
  if (!pyr || !d_pts || !d_rects || batch < 0 || n_pts < 1 || rect_stride < 4 || max_flow < 0 || pyr->levels < 1 ||
      pyr->levels > AGT_MAX_LEVELS)
    AGT_FAIL(ctx, AGT_ERR_INVALID, "agt_lk_rects: bad arguments");
  lk_rects_kernel<<<(batch + 3) / 4, 128, 0, ctx->stream>>>(d_pts, d_valid, n_pts, pyr->width[0], pyr->height[0], pyr->levels - 1,
                                                            max_flow, d_rects, rect_stride, batch);
  AGT_LAUNCH_CHECK(ctx);
  return AGT_OK;
}

static int lk_impl(agt_ctx* ctx, const agt_pyramid* prev, const agt_pyramid* next, const float* d_prev_pts, float* d_next_pts,
                   uint8_t* d_status, float* d_err, int batch, int n_pts, const int32_t* d_n_tags, const int32_t* d_rects_prev,
                   const int32_t* d_rects_next, int rect_stride, const uint8_t* d_mask, uint8_t* d_left_roi) {
  if (!prev || !next || batch < 0 || n_pts < 0) AGT_FAIL(ctx, AGT_ERR_INVALID, "agt_lk: null pyramid or negative size");
  if ((int64_t)batch * n_pts > 0 && (!d_prev_pts || !d_next_pts || !d_status || !d_err))
    AGT_FAIL(ctx, AGT_ERR_INVALID, "agt_lk: null point / status / err buffer");
  if (prev->levels < 1 || prev->levels > AGT_MAX_LEVELS || prev->levels != next->levels)
    AGT_FAIL(ctx, AGT_ERR_INVALID, "agt_lk: pyramids must have the same 1..%d levels", AGT_MAX_LEVELS);
  for (int l = 0; l < prev->levels; ++l)
    if (prev->width[l] != next->width[l] || prev->height[l] != next->height[l])
      AGT_FAIL(ctx, AGT_ERR_INVALID, "agt_lk: prev/next level %d sizes differ", l);
  int64_t total = (int64_t)batch * n_pts;
  if (total == 0) return AGT_OK;
  int64_t blocks = (total + WARPS_PER_CTA - 1) / WARPS_PER_CTA;
  if (blocks > 0x7fffffffLL) AGT_FAIL(ctx, AGT_ERR_INVALID, "agt_lk: batch too large");
  // (agt_lk_fallback skips the frames that kept their detections - nearly all: their CTAs leave at once - so it may be 8 x larger)
  if (!d_rects_prev && !d_rects_next && !d_mask && prev->levels > 1 && total <= (int64_t)ctx->lk_split_max * (d_n_tags ? 8 : 1)) {
    // few corners (a frame-step of the stream pipeline): the caller waits for the slowest corner, so a warp per level
    const int smem = prev->levels * (int)sizeof(WarpSmem);
    lk_levels_kernel<<<(unsigned)total, prev->levels * 32, smem, ctx->stream>>>(*prev, *next, d_prev_pts, d_next_pts, d_status, d_err, n_pts,
                                                                              d_n_tags);
    AGT_LAUNCH_CHECK(ctx);
    return AGT_OK;
  }
  const bool stride = d_mask != nullptr && blocks > 8LL * ctx->sm_count;
  if (stride) blocks = 8LL * ctx->sm_count;      // warps stride over the corners
  const bool roi = d_rects_prev || d_rects_next;
  constexpr int kSmem = WARPS_PER_CTA * (int)sizeof(WarpSmem);
  static bool attr_set[64] = {false};
  if (!attr_set[ctx->device & 63]) {
    AGT_CUDA(ctx, cudaFuncSetAttribute(lk_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmem));
    AGT_CUDA(ctx, cudaFuncSetAttribute(lk_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmem));
    AGT_CUDA(ctx, cudaFuncSetAttribute(lk_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmem));
    AGT_CUDA(ctx, cudaFuncSetAttribute(lk_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmem));
    attr_set[ctx->device & 63] = true;
  }
#define AGT_LK_LAUNCH(R, S)                                                                                                     \
  lk_kernel<R, S><<<(unsigned)blocks, WARPS_PER_CTA * 32, kSmem, ctx->stream>>>(*prev, *next, d_prev_pts, d_next_pts, d_status, d_err, \
                                                                            n_pts, total, d_n_tags, d_rects_prev, d_rects_next,   \
                                                                            rect_stride, d_mask, d_left_roi)
  if (roi) { if (stride) AGT_LK_LAUNCH(true, true); else AGT_LK_LAUNCH(true, false); }
  else     { if (stride) AGT_LK_LAUNCH(false, true); else AGT_LK_LAUNCH(false, false); }
#undef AGT_LK_LAUNCH
  AGT_LAUNCH_CHECK(ctx);
  return AGT_OK;
}
