// Region-of-interest plan of one dense refinement, shared by the kernel (thread 0 of the CTA) and by
// the host entry point agt_refine_host (which uploads only the rectangle the kernel can touch).
// Everything is float64 and depends only on the initial pose, the camera and the model radius, so
// host and device arrive at the same integers (a last-ulp difference in atan/tan between host and device libm
// could move an edge by one pixel; the upload rectangle carries a >= 2 px halo and frames that read outside
// what was uploaded are detected and redone, so this cannot change results).
#pragma once
#include "agt_common.cuh"

constexpr int AGT_DPR_TILE_ROWS = 270;
constexpr int AGT_DPR_TILE_PITCH = 288;          // 272 + 16 B alignment slack; 2 CTAs of 76.5 KB per SM
constexpr int AGT_DPR_DRIFT_MARGIN = 8;          // level pixels the projection may drift during LM

struct agt_dpr_plan {
  int level;
  int rx0, ry0, rx1, ry1;   // predicted ROI at `level` (bounding sphere + margin), clamped to the level, rx0 % 16 == 0
  int tx0, ty0, tw, th;     // staged tile: the ROI cut to the shared-memory capacity
};

__host__ __device__ inline agt_dpr_plan agt_make_dpr_plan(const agt_camera& cam, double pitch, double radius,
                                                          const double t[3], const int32_t* widths,
                                                          const int32_t* heights, int levels) {
  agt_dpr_plan p;
  double q = cam.fx * pitch / t[2];
  int lvl = q < 2.0 ? 0 : (q < 4.0 ? 1 : (q < 8.0 ? 2 : 3));
  if (!(t[2] > 0.0)) lvl = 0;
  if (lvl > levels - 1) lvl = levels - 1;
  p.level = lvl;
  const int lw = widths[lvl], lh = heights[lvl];
  const double sc = 1.0 / (double)(1 << lvl);
  // exact image extent of the bounding sphere (centre t, radius `radius`): in the x-z plane the tangent rays
  // make angles atan(x/z) +- asin(r/|(x,z)|) with the optical axis; likewise in y-z
  const double margin = AGT_DPR_DRIFT_MARGIN + 2;
  double zc = t[2] > 1e-6 ? t[2] : 1e-6;
  double ext[4];
  for (int a = 0; a < 2; ++a) {
    double c = t[a], f = a == 0 ? cam.fx : cam.fy, pp = a == 0 ? cam.cx : cam.cy;
    double d = sqrt(c * c + zc * zc);
    double sb = radius / d;
    if (sb > 0.95) sb = 0.95;                       // camera (almost) inside the sphere: huge ROI, clamped below
    double al = atan2(c, zc), be = asin(sb);
    double lo_a = al - be, hi_a = al + be;
    if (lo_a < -1.5) lo_a = -1.5;
    if (hi_a > 1.5) hi_a = 1.5;
    ext[2 * a] = (f * tan(lo_a) + pp) * sc - margin;
    ext[2 * a + 1] = (f * tan(hi_a) + pp) * sc + margin;
  }
  double lo = -1e6, hi = 1e6;
  double fx0 = floor(ext[0]), fy0 = floor(ext[2]), fx1 = ceil(ext[1]) + 1, fy1 = ceil(ext[3]) + 1;
  if (!(fx0 == fx0)) fx0 = hi;          // NaN pose: empty ROI
  if (!(fy0 == fy0)) fy0 = hi;
  if (!(fx1 == fx1)) fx1 = lo;
  if (!(fy1 == fy1)) fy1 = lo;
  fx0 = fx0 < lo ? lo : (fx0 > hi ? hi : fx0); fy0 = fy0 < lo ? lo : (fy0 > hi ? hi : fy0);
  fx1 = fx1 < lo ? lo : (fx1 > hi ? hi : fx1); fy1 = fy1 < lo ? lo : (fy1 > hi ? hi : fy1);
  int x0 = (int)fx0, y0 = (int)fy0, x1 = (int)fx1, y1 = (int)fy1;
  x0 = (x0 > 0 ? x0 : 0) & ~15; y0 = y0 > 0 ? y0 : 0;
  x1 = x1 < lw ? x1 : lw; y1 = y1 < lh ? y1 : lh;
  if (x1 < x0) x1 = x0;
  if (y1 < y0) y1 = y0;
  p.rx0 = x0; p.ry0 = y0; p.rx1 = x1; p.ry1 = y1;
  int tw = x1 - x0, th = y1 - y0;
  if (tw > AGT_DPR_TILE_PITCH) { int cut = (tw - AGT_DPR_TILE_PITCH + 31) / 32 * 16; x0 += cut; tw = lw - x0 < AGT_DPR_TILE_PITCH ? lw - x0 : AGT_DPR_TILE_PITCH; }
  if (th > AGT_DPR_TILE_ROWS) { y0 += (th - AGT_DPR_TILE_ROWS) / 2; th = AGT_DPR_TILE_ROWS; }
  p.tx0 = x0; p.ty0 = y0; p.tw = tw > 0 ? tw : 0; p.th = th > 0 ? th : 0;
  return p;
}

// Level-0 rectangle (x0,y0,x1,y1; x multiples of 16) the refinements of one frame can read: union over its
// hypotheses of the predicted ROI scaled to level 0 plus the pyrDown halo of the chain down to the level used.
// Returns false (and an empty rectangle) if no hypothesis projects into the frame.
__host__ __device__ inline bool agt_dpr_rect_l0(const agt_camera& cam, double pitch, double radius, const double* init,
                                                int n_hyp, const int32_t* widths, const int32_t* heights, int levels,
                                                int32_t rect[4]) {
  const int W = widths[0], H = heights[0];
  int x0 = W, y0 = H, x1 = 0, y1 = 0;
  for (int hyp = 0; hyp < n_hyp; ++hyp) {
    const double* p = init + hyp * 6;
    agt_dpr_plan plan = agt_make_dpr_plan(cam, pitch, radius, p + 3, widths, heights, levels);
    if (plan.rx1 <= plan.rx0 || plan.ry1 <= plan.ry0) continue;
    const int l = plan.level, pad = 2 << l;
    int a = (plan.rx0 << l) - pad, b = (plan.ry0 << l) - pad;
    int c = ((plan.rx1 - 1) << l) + pad + 1, d = ((plan.ry1 - 1) << l) + pad + 1;
    x0 = a < x0 ? a : x0; y0 = b < y0 ? b : y0; x1 = c > x1 ? c : x1; y1 = d > y1 ? d : y1;
  }
  x0 = (x0 > 0 ? x0 : 0) & ~15; y0 = y0 > 0 ? y0 : 0;
  x1 = (x1 + 15) & ~15; x1 = x1 < W ? x1 : W; y1 = y1 < H ? y1 : H;
  bool ok = x1 > x0 && y1 > y0;
  rect[0] = ok ? x0 : 0; rect[1] = ok ? y0 : 0; rect[2] = ok ? x1 : 0; rect[3] = ok ? y1 : 0;
  return ok;
}
