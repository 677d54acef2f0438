// K4: dense pose refinement - batched photometric Levenberg-Marquardt that never
// leaves the device.  One CTA per (frame, hypothesis).
//
// No reference code exists for this stage (README.md:20 names it as future work);
// the executable specification is oracle/dpr_oracle.py (SURVEY.md 8a row A6, 9.4):
// visibility and pyramid level frozen at the initial pose; per sample a pinhole
// projection, bilinear intensity and bilinear Scharr gradient of level l, residual
// r = I - O, 1x6 Jacobian [Y x g, g] for the left perturbation R <- exp(w) R;
// H = J^T J (21), b = J^T r (6), c = 1/2 sum r^2; LM with lambda*diag(H), accept
// iff the cost decreases, stop rules as in the oracle.
//
// B200 mapping: the level-l region of interest (<= 272x272 u8, the projected
// bounding sphere plus a drift margin) is staged ONCE per CTA into shared memory
// with 128-bit loads and reused by every LM evaluation, so HBM sees each ROI byte
// once per refinement; no gradient plane is materialised - the 4x4 u8 footprint of
// a sample is fetched with two aligned 32-bit shared loads + a byte permute per
// row and the four Scharr values come from 16 dp4a.  The projection of a sample
// runs in float64 (see the note in the sample loop), intensity / gradient /
// Jacobian in float32; the 28 sums are reduced by warp shuffles and across warps in float64
// (the cost in float64 from the start); one thread runs the 6x6 Cholesky / LM
// bookkeeping in float64.  Samples whose footprint leaves the staged tile fall
// back to global loads, so results do not depend on the tile size.
#include <cooperative_groups.h>
#include <cstddef>

#include "agt_dpr_plan.cuh"
#include "agt_pyr_stream.cuh"

namespace cg = cooperative_groups;

namespace {

constexpr int DPR_THREADS = 256;
constexpr int DPR_WARPS = DPR_THREADS / 32;
constexpr int TILE_ROWS = AGT_DPR_TILE_ROWS;
constexpr int TILE_PITCH = AGT_DPR_TILE_PITCH;
constexpr int TILE_BYTES = TILE_ROWS * TILE_PITCH + 16;   // +16: the unaligned fetch reads one word past its window
// fused K1: scratch of the CTA-level pyrDown that builds the level-l ROI inside the refinement kernel
constexpr int PB_ROWS = 8;                        // output rows per band
constexpr int PB_IN_ROWS = 2 * PB_ROWS + 3;       // input rows a band reads
constexpr int PB_OUT_W = 288;                     // output columns per panel (the widest tile)
constexpr int PB_IN_PITCH = 2 * PB_OUT_W + 32;    // staged input row: 16 B of halo room on each side
constexpr int PB_H_PITCH = PB_OUT_W;              // horizontal-pass row, uint16 elements
constexpr int PB_BYTES = 2 * PB_IN_ROWS * PB_IN_PITCH + PB_IN_ROWS * PB_H_PITCH * 2;   // two input buffers (the next band is prefetched)
// 1: project the samples in float32 (see the sample loop); 0: the float64 projection of round 1
#ifndef AGT_DPR_F32_PROJECTION
#define AGT_DPR_F32_PROJECTION 1
#endif
constexpr int NSUM = 28;                   // 21 H + 6 b + (cost kept separately in double) + count
constexpr double COS_VISIBLE = 0.25881904510252074;   // cos 75 deg
constexpr double LAMBDA0 = 1e-3, LAMBDA_MIN = 1e-9, LAMBDA_MAX = 1e6;
constexpr int MAX_EVALS = 50;
constexpr double TOL_ROT = 5e-6, TOL_TRANS = 1e-6;
// Aitken step length (oracle/dpr_oracle.py): consecutive Gauss-Newton steps are collinear, their ratio gives the contraction
constexpr double AITKEN_COS2 = 0.64, AITKEN_QMAX = 0.75, ALPHA_MIN = 0.25, ALPHA_MAX = 4.0;
// a trial pose is accepted unless the cost rises by more than this fraction (oracle/dpr_oracle.py: the Scharr gradient is not
// the exact derivative of the bilinear interpolant, so near convergence the cost moves by ~1e-5 of itself either way; the
// slack lets the loop contract onto J^T r = 0 instead of stalling where that noise first rejects a step); no trial above the
// cost at the initial pose is accepted, so that the slack cannot compound into a run that ends worse than it started
constexpr double ACCEPT_SLACK = 1e-2;

struct DprShared {
  // trial pose: float64 for the projection, float32 for the Jacobian
  __align__(16) double Rd[12];   // level-l projection matrix of the trial pose, K_l [R | t] with K_l = [[fx_l 0 cx_l] [0 fy_l cy_l] [0 0 1]]:
                                 // rows as R-part (9, row-major) then t-part (3); six 128-bit broadcast loads per sample
  double Pt[12];                 // trial pose itself: rotation (row-major) + translation
  __align__(16) float Rf[12];    // (R0,R3) (R1,R4) (R2,R5) (t0,t1) as pairs for the packed float32 ops, then R6 R7 R8 t2
  __align__(16) double proj[4];  // fx*2^-l, fy*2^-l, cx*2^-l, cy*2^-l (two 128-bit loads)
  float fx, fy;
  float gscale;          // 2^-level / 32
  int level, lw, lh;
  int64_t lpitch;
  const uint8_t* limg;   // level image of this frame
  int tx0, ty0, tw, th;  // staged tile: origin (level px), size
  int xbias, ybias;      // high word of (1.5 * 2^20 + tile origin + 1): see the sample loop
  float projf[4];        // fx, fy, cx, cy of level l in float32
  uint32_t tw_m3, th_m3; // tile size - 3 (0 for a tile smaller than one footprint)
  int rx0, ry0, rx1, ry1;   // predicted ROI (see agt_dpr_plan)
  int left_roi;          // a sample footprint left the predicted ROI at some evaluation
  int n_active;
  int act_begin[AGT_MAX_TAGS];   // first sample of each active tag
  int act_prefix[AGT_MAX_TAGS + 1];
  int stop;
  int zero;              // 0, read at run time (an ordering dependency the compiler cannot fold away)
  double wsum[DPR_WARPS][NSUM + 2];
  double tot[2][NSUM + 2];  // cluster exchange only, double-buffered by evaluation parity
  // LM state, touched by warp 0 only (kept out of registers)
  double Pc[12];         // accepted pose: rotation (row-major) + translation
  double Hb[27];         // normal equations at the accepted pose: H (21, packed upper triangle by rows) + b (6)
  double dstep[6], cc, lam;   // dstep: the applied step alpha * d of the pending trial
  double c0;             // cost at the initial pose: the bound of every accepted cost
  double dgn[6], dprev[6], alpha;   // solve's step of the pending trial / of the last accepted one (Aitken step length)
  int have_prev;
  int nc, evals, status;
};

// Two CTAs per SM: dynamic + static shared memory + the 1 KB the driver reserves per CTA must fit half of the 228 KB of an
// SM.  (Round 2 found this the hard way: 96 bytes of new LM state left one CTA per SM and made the kernel 1.5x slower.)
static_assert(2 * (TILE_BYTES + PB_BYTES + (int)sizeof(DprShared) + 1024) <= 233472, "dpr_kernel must keep 2 CTAs per SM");

// (L2-coherent loads: with K1 fused the level image is written by this very launch, so the read-only path is out)
__device__ __forceinline__ uint32_t ld4_global(const uint8_t* p) {
  return (uint32_t)__ldcg(p) | ((uint32_t)__ldcg(p + 1) << 8) | ((uint32_t)__ldcg(p + 2) << 16) | ((uint32_t)__ldcg(p + 3) << 24);
}

// ---- packed float32 pairs (sm_100 FFMA2 / FMUL2 / FADD2: two lanes per issue slot) --------------------------
// The sample loop is bound by instruction issue, not by any one pipe, so everything that comes in (x, y)
// pairs - the rotated lever arm, the (gx, gy) gradient taps, the normal-equation products - runs packed.
// ptxas folds scalar broadcasts and lane swaps into the operand modifiers (R.F32, R.F32x2.LO_HI).
typedef unsigned long long f32x2;
__device__ __forceinline__ f32x2 pk2(float lo, float hi) { f32x2 r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi)); return r; }
__device__ __forceinline__ f32x2 pk2(int lo, int hi) { f32x2 r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "r"(lo), "r"(hi)); return r; }
__device__ __forceinline__ float lo2(f32x2 v) { float a; asm("{ .reg .b32 t; mov.b64 {%0, t}, %1; }" : "=f"(a) : "l"(v)); return a; }
__device__ __forceinline__ float hi2(f32x2 v) { float b; asm("{ .reg .b32 t; mov.b64 {t, %0}, %1; }" : "=f"(b) : "l"(v)); return b; }
__device__ __forceinline__ f32x2 bc2(float s) { return pk2(s, s); }
__device__ __forceinline__ f32x2 swap2(f32x2 v) { return pk2(hi2(v), lo2(v)); }
__device__ __forceinline__ f32x2 fma2(f32x2 a, f32x2 b, f32x2 c) { f32x2 d; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c)); return d; }
__device__ __forceinline__ f32x2 mul2(f32x2 a, f32x2 b) { f32x2 d; asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }
__device__ __forceinline__ f32x2 add2(f32x2 a, f32x2 b) { f32x2 d; asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }

// d = acc + sum_k px.byte[k] (unsigned) * coef.byte[k] (signed)
__device__ __forceinline__ int dp4c(uint32_t px, int coef, int acc) {
  int d;
  asm("dp4a.u32.s32 %0, %1, %2, %3;" : "=r"(d) : "r"(px), "r"(coef), "r"(acc));
  return d;
}

// ---- serial LM phase helpers (one thread per CTA runs them while 255 wait: keep the dependency chains short) ----
// exp([w]x) for an LM step: Taylor series of sin(t)/t and (1-cos t)/t^2 in t^2 for |w| < 0.5 (truncation < 1e-16),
// libm sincos otherwise
__device__ __forceinline__ void rodrigues_step(const double w[3], double R[9]) {
  const double t2 = w[0] * w[0] + w[1] * w[1] + w[2] * w[2];
  if (t2 >= 0.25) { agt_rodrigues(w, R); return; }
  double a = 1.0 / 6227020800.0, b = 1.0 / 87178291200.0;
  a = fma(a, t2, -1.0 / 39916800.0); b = fma(b, t2, -1.0 / 479001600.0);
  a = fma(a, t2, 1.0 / 362880.0);    b = fma(b, t2, 1.0 / 3628800.0);
  a = fma(a, t2, -1.0 / 5040.0);     b = fma(b, t2, -1.0 / 40320.0);
  a = fma(a, t2, 1.0 / 120.0);       b = fma(b, t2, 1.0 / 720.0);
  a = fma(a, t2, -1.0 / 6.0);        b = fma(b, t2, -1.0 / 24.0);
  a = fma(a, t2, 1.0);               b = fma(b, t2, 0.5);
  const double c = 1.0 - b * t2;
  R[0] = c + b * w[0] * w[0];        R[1] = b * w[0] * w[1] - a * w[2]; R[2] = b * w[0] * w[2] + a * w[1];
  R[3] = b * w[1] * w[0] + a * w[2]; R[4] = c + b * w[1] * w[1];        R[5] = b * w[1] * w[2] - a * w[0];
  R[6] = b * w[2] * w[0] - a * w[1]; R[7] = b * w[2] * w[1] + a * w[0]; R[8] = c + b * w[2] * w[2];
}

// shared-window address kept opaque so that it stays in one register instead of being re-derived in the loop;
// the loads below carry a memory clobber so that the compiler keeps (and orders) the C++ stores they read
__device__ __forceinline__ uint32_t smem_addr(const void* p) {
  uint32_t a = (uint32_t)__cvta_generic_to_shared(p), o;
  asm volatile("mov.u32 %0, %1;" : "=r"(o) : "r"(a));
  return o;
}
__device__ __forceinline__ double2 lds_f64x2(uint32_t a) {
  double2 v;
  asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(v.x), "=d"(v.y) : "r"(a) : "memory");
  return v;
}
__device__ __forceinline__ uint32_t lds_u32(uint32_t a) {
  uint32_t v;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a) : "memory");
  return v;
}

// thread 0 publishes a trial pose to the sample loop
__device__ __forceinline__ void publish_pose(DprShared& S, const double* R, const double* t) {
  const double fxl = S.proj[0], fyl = S.proj[1], cxl = S.proj[2], cyl = S.proj[3];
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    S.Rd[c] = fma(fxl, R[c], cxl * R[6 + c]);
    S.Rd[3 + c] = fma(fyl, R[3 + c], cyl * R[6 + c]);
    S.Rd[6 + c] = R[6 + c];
  }
  S.Rd[9] = fma(fxl, t[0], cxl * t[2]);
  S.Rd[10] = fma(fyl, t[1], cyl * t[2]);
  S.Rd[11] = t[2];
#pragma unroll
  for (int i = 0; i < 9; ++i) S.Pt[i] = R[i];
#pragma unroll
  for (int i = 0; i < 3; ++i) S.Pt[9 + i] = t[i];
#pragma unroll
  for (int c = 0; c < 3; ++c) { S.Rf[2 * c] = (float)R[c]; S.Rf[2 * c + 1] = (float)R[3 + c]; S.Rf[8 + c] = (float)R[6 + c]; }
  S.Rf[6] = (float)t[0]; S.Rf[7] = (float)t[1]; S.Rf[11] = (float)t[2];
}

// packed signed-byte coefficient words (little endian: byte 0 multiplies the left-most pixel)
constexpr int C_DX0_3 = (int)0x000300FD;    // ( -3,  0,  3,  0)   horizontal difference at x0, row weight 3
constexpr int C_DX0_10 = (int)0x000A00F6;   // (-10,  0, 10,  0)   ... row weight 10
constexpr int C_DX1_3 = (int)0x0300FD00;    // (  0, -3,  0,  3)   horizontal difference at x0+1
constexpr int C_DX1_10 = (int)0x0A00F600;   // (  0,-10,  0, 10)
constexpr int C_SM0 = (int)0x00030A03;      // (  3, 10,  3,  0)   horizontal smoothing at x0
constexpr int C_SM1 = (int)0x030A0300;      // (  0,  3, 10,  3)   horizontal smoothing at x0+1
constexpr int C_SM0_NEG = (int)0x00FDF6FD;  // ( -3,-10, -3,  0)
constexpr int C_SM1_NEG = (int)0xFDF6FD00;  // (  0, -3,-10, -3)
__constant__ int kCoef[8] = {C_DX0_3, C_DX0_10, C_DX1_3, C_DX1_10, C_SM0, C_SM1, C_SM0_NEG, C_SM1_NEG};

// Per-refinement setup that depends only on the initial pose, computed by one thread per refinement in a launch of its
// own (dpr_prep_kernel) instead of by thread 0 of every CTA while 255 threads wait: pyramid level and ROI plan
// (atan / asin / tan), rotation matrix of the initial pose (sincos) and the visibility test of each tag.
struct __align__(16) DprJob {
  int32_t level, rx0, ry0, rx1;       // 16-byte words read by every thread of the CTA
  int32_t ry1, tx0, ty0, tw;
  int32_t th;
  uint32_t active;                    // bit k: tag k passes the visibility test at the initial pose
  int32_t pad[2];
  double R[9];                        // rotation of the initial pose, row-major
  double pad2;
};
static_assert(sizeof(DprJob) == 128, "DprJob layout");

// tag k passes the visibility test at the pose (Rc, tc): its normal makes less than 75 degrees with the ray to its centre
__device__ __forceinline__ bool dpr_tag_visible(const agt_model& model, const double Rc[9], const double tc[3], int k) {
  double c[3], n[3];
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    c[i] = Rc[i * 3] * model.centres[k][0] + Rc[i * 3 + 1] * model.centres[k][1] + Rc[i * 3 + 2] * model.centres[k][2] + tc[i];
    n[i] = Rc[i * 3] * model.normals[k][0] + Rc[i * 3 + 1] * model.normals[k][1] + Rc[i * 3 + 2] * model.normals[k][2];
  }
  const double cn = sqrt(c[0] * c[0] + c[1] * c[1] + c[2] * c[2]);
  const double d = -(n[0] * c[0] + n[1] * c[1] + n[2] * c[2]) / cn;
  return d > COS_VISIBLE;
}

__device__ __forceinline__ void dpr_fill_job(DprJob& j, const agt_dpr_plan& plan, uint32_t active, const double Rc[9]) {
  j.level = plan.level; j.rx0 = plan.rx0; j.ry0 = plan.ry0; j.rx1 = plan.rx1; j.ry1 = plan.ry1;
  j.tx0 = plan.tx0; j.ty0 = plan.ty0; j.tw = plan.tw; j.th = plan.th; j.active = active; j.pad[0] = j.pad[1] = 0;
#pragma unroll
  for (int i = 0; i < 9; ++i) j.R[i] = Rc[i];
  j.pad2 = 0.0;
}

__global__ void dpr_prep_kernel(agt_pyramid pyr, agt_camera cam, agt_model model, const double* __restrict__ init, int n_hyp,
                                const uint8_t* __restrict__ mask, DprJob* __restrict__ jobs, int64_t n_jobs) {
  const int64_t job = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (job >= n_jobs) return;
  if (mask != nullptr && mask[job / n_hyp] == 0) return;
  const double* p0 = init + job * 6;
  const double r0[3] = {p0[0], p0[1], p0[2]}, tc[3] = {p0[3], p0[4], p0[5]};
  double Rc[9];
  agt_rodrigues(r0, Rc);
  const agt_dpr_plan plan = agt_make_dpr_plan(cam, model.pitch, model.radius, tc, pyr.width, pyr.height, pyr.levels);
  uint32_t active = 0;
  for (int k = 0; k < model.n_tags; ++k)
    if (dpr_tag_visible(model, Rc, tc, k)) active |= 1u << k;
  DprJob j;
  dpr_fill_job(j, plan, active, Rc);
  jobs[job] = j;
}

// The same setup by one warp of the refinement's own CTA (cluster launches: a batch smaller than the machine is a chain of
// dependent launches per frame-step, and a setup launch of its own is a tenth of that chain): every lane derives the rotation
// and the ROI plan, lane k tests tag k, lane 0 writes the record.  Every CTA of a cluster arrives at the same record.
__device__ __forceinline__ void dpr_prep_warp(const agt_pyramid& pyr, const agt_camera& cam, const agt_model& model,
                                              const double* __restrict__ p0, DprJob* out, int lane) {
  const double r0[3] = {p0[0], p0[1], p0[2]}, tc[3] = {p0[3], p0[4], p0[5]};
  double Rc[9];
  agt_rodrigues(r0, Rc);
  const agt_dpr_plan plan = agt_make_dpr_plan(cam, model.pitch, model.radius, tc, pyr.width, pyr.height, pyr.levels);
  uint32_t active = 0;
  for (int k0 = 0; k0 < model.n_tags; k0 += 32) {
    const int k = k0 + lane;
    const bool vis = k < model.n_tags && dpr_tag_visible(model, Rc, tc, k < model.n_tags ? k : 0);
    active |= __ballot_sync(0xffffffffu, vis) << k0;
  }
  if (lane == 0) dpr_fill_job(*out, plan, active, Rc);
  __syncwarp();
}
// BORDER_REFLECT_101 index: in range almost always, the general fold otherwise
__device__ __forceinline__ int reflect101(int i, int n) { return (unsigned)i < (unsigned)n ? i : agt_reflect101(i, n); }

// cv2.pyrDown of one rectangle of a level, by the whole CTA: out = (sum 5x5 [1 4 6 4 1]^2 in + 128) >> 8, integer, so the
// result is bit-identical to K1 whatever the order.  Output rectangle [x0,x1) x [y0,y1) in destination pixels, x0 % 16 == 0,
// inside the destination level.  Bands of PB_ROWS output rows: the 2*rows+3 input rows are staged with 16-byte asynchronous
// copies (reflected borders patched in shared memory), a horizontal pass leaves packed uint16 sums (8 dp4a per 4 outputs),
// a vertical pass on uint16 pairs (16 * 4080 + 128 fits) writes 4 output bytes per thread to the global level and, where it
// overlaps, to the shared-memory tile of the refinement.
__device__ void cta_pyr_down_region(const uint8_t* __restrict__ src, int sw, int sh, int64_t spitch, uint8_t* __restrict__ dst,
                                    int64_t dpitch, uint8_t* tile, int tx0, int ty0, int tw, int th, int x0, int y0, int x1,
                                    int y1, uint8_t* s_in, uint16_t* s_h) {
  const int tid = threadIdx.x;
  const bool vec = ((spitch & 15) == 0) && ((reinterpret_cast<uintptr_t>(src) & 15) == 0);
  const bool dvec = ((dpitch & 3) == 0) && ((reinterpret_cast<uintptr_t>(dst) & 3) == 0);
  const uint32_t s_in_a = (uint32_t)__cvta_generic_to_shared(s_in);
  const int n_bands = (y1 - y0 + PB_ROWS - 1) / PB_ROWS, n_panels = (x1 - x0 + PB_OUT_W - 1) / PB_OUT_W;
  const int n_items = n_bands * n_panels;
  // geometry of work item i (a band of a panel) and the request for its input rows into buffer i & 1
  auto stage = [&](int i) {
    if (i < n_items) {
      const int px0 = x0 + (i / n_bands) * PB_OUT_W, oy0 = y0 + (i % n_bands) * PB_ROWS;
      const int pw = min(PB_OUT_W, (x1 - px0 + 3) & ~3);
      const int in_c0 = 2 * px0 - 16, in_chunks = (2 * pw + 32) >> 4;      // source column of staged offset 0 (16 B aligned)
      const int in_rows = 2 * min(PB_ROWS, y1 - oy0) + 3, iy0 = 2 * oy0 - 2;
      uint8_t* buf = s_in + (i & 1) * (PB_IN_ROWS * PB_IN_PITCH);
      const uint32_t buf_a = s_in_a + (i & 1) * (PB_IN_ROWS * PB_IN_PITCH);
      for (int r = tid >> 5; r < in_rows; r += DPR_WARPS)
      for (int c = tid & 31; c < in_chunks; c += 32) {      // a warp per row, a lane per 16-byte chunk (no divisions)
        const int col = in_c0 + 16 * c;
        const uint8_t* g = src + (int64_t)reflect101(iy0 + r, sh) * spitch + col;
        if (col >= 0 && col + 16 <= (int)spitch) {
          if (vec) {
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" :: "r"(buf_a + r * PB_IN_PITCH + 16 * c), "l"(g) : "memory");
          } else {
            for (int q = 0; q < 16; ++q) buf[r * PB_IN_PITCH + 16 * c + q] = __ldcg(g + q);
          }
        } else {
          for (int q = 0; q < 16; ++q) {
            const int cc = col + q;
            buf[r * PB_IN_PITCH + 16 * c + q] = (cc >= 0 && cc < sw) ? __ldcg(g + q) : (uint8_t)0;
          }
        }
      }
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
  };
  stage(0);
  for (int i = 0; i < n_items; ++i) {
    stage(i + 1);                                        // the next band travels while this one is computed
    asm volatile("cp.async.wait_group 1;" ::: "memory");
    __syncthreads();
    const int px0 = x0 + (i / n_bands) * PB_OUT_W, oy0 = y0 + (i % n_bands) * PB_ROWS;
    const int pw = min(PB_OUT_W, (x1 - px0 + 3) & ~3), quads = pw >> 2;
    const int in_c0 = 2 * px0 - 16;
    const int rows = min(PB_ROWS, y1 - oy0), in_rows = 2 * rows + 3;
    uint8_t* buf = s_in + (i & 1) * (PB_IN_ROWS * PB_IN_PITCH);
    // ---- reflected columns: -2, -1 on the left edge of the level, sw .. on the right edge ----
    {
      const int c_lo = 2 * px0 - 2, c_hi = 2 * (px0 + pw - 1) + 2;        // tap range of this panel
      const int n_left = c_lo < 0 ? -c_lo : 0, n_right = c_hi >= sw ? c_hi - sw + 1 : 0;
      if (n_left + n_right > 0) {
        for (int k = tid; k < in_rows * (n_left + n_right); k += DPR_THREADS) {
          const int r = k / (n_left + n_right), q = k - r * (n_left + n_right);
          const int cc = q < n_left ? c_lo + q : sw + (q - n_left);
          buf[r * PB_IN_PITCH + (cc - in_c0)] = buf[r * PB_IN_PITCH + (reflect101(cc, sw) - in_c0)];
        }
        __syncthreads();
      }
    }
    // ---- horizontal pass: 4 outputs from 4 words ----
    for (int r = tid >> 5; r < in_rows; r += DPR_WARPS)
    for (int q = tid & 31; q < quads; q += 32) {
      const uint32_t* w = reinterpret_cast<const uint32_t*>(buf + r * PB_IN_PITCH + 12 + 8 * q);      // bytes 2*ox-4 ..
      const uint32_t w0 = w[0], w1 = w[1], w2 = w[2], w3 = w[3];
      const int h0 = dp4c(w1, 0x00010406, dp4c(w0, 0x04010000, 0));      // taps at bytes 2..6
      const int h1 = dp4c(w2, 0x00000001, dp4c(w1, 0x04060401, 0));      // bytes 4..8
      const int h2 = dp4c(w2, 0x00010406, dp4c(w1, 0x04010000, 0));      // bytes 6..10
      const int h3 = dp4c(w3, 0x00000001, dp4c(w2, 0x04060401, 0));      // bytes 8..12
      *reinterpret_cast<uint2*>(s_h + r * PB_H_PITCH + 4 * q) = make_uint2((uint32_t)h0 | ((uint32_t)h1 << 16), (uint32_t)h2 | ((uint32_t)h3 << 16));
    }
    __syncthreads();
    // ---- vertical pass on uint16 pairs ----
    for (int r = tid >> 5; r < rows; r += DPR_WARPS)
    for (int q = tid & 31; q < quads; q += 32) {
      const uint2* hp = reinterpret_cast<const uint2*>(s_h + (2 * r) * PB_H_PITCH + 4 * q);
      const uint2 a = hp[0], b = hp[PB_H_PITCH / 4], c = hp[2 * (PB_H_PITCH / 4)], d = hp[3 * (PB_H_PITCH / 4)], e = hp[4 * (PB_H_PITCH / 4)];
      const uint32_t v0 = a.x + e.x + 4u * (b.x + d.x) + 6u * c.x + 0x00800080u;
      const uint32_t v1 = a.y + e.y + 4u * (b.y + d.y) + 6u * c.y + 0x00800080u;
      const uint32_t out = __byte_perm(v0, v1, 0x7531);                  // the high byte of each uint16
      const int ox = px0 + 4 * q, oy = oy0 + r;
      if (dvec && ox + 4 <= (int)dpitch) {
        *reinterpret_cast<uint32_t*>(dst + (int64_t)oy * dpitch + ox) = out;
      } else {
        for (int m = 0; m < 4; ++m)
          if (ox + m < (int)dpitch) dst[(int64_t)oy * dpitch + ox + m] = (uint8_t)(out >> (8 * m));
      }
      if (tile != nullptr && oy >= ty0 && oy < ty0 + th && ox >= tx0 && ox < tx0 + tw)
        *reinterpret_cast<uint32_t*>(tile + (oy - ty0) * TILE_PITCH + (ox - tx0)) = out;
    }
    __syncthreads();                                     // s_h and buffer i & 1 are free again
  }
  asm volatile("cp.async.wait_all;" ::: "memory");
}

// kCluster > 1: a thread-block cluster of kCluster CTAs shares one refinement.  Used when the batch is smaller than
// the machine (camera streams: one pose per stream per step): every CTA stages the ROI, takes every kCluster-th
// slice of the samples, every CTA reads every CTA's partial sums through distributed shared memory and takes the
// (identical) LM step itself.  One cluster barrier per evaluation.
template <int kCluster>
__global__ void __launch_bounds__(DPR_THREADS, 2)
dpr_kernel(agt_pyramid pyr, agt_camera cam, const float4* __restrict__ samples, agt_model model,
           const double* __restrict__ init, int n_hyp, const uint8_t* __restrict__ mask, double* __restrict__ pose_out, float* __restrict__ cost_out,
           int32_t* __restrict__ nvalid_out, int32_t* __restrict__ evals_out, uint8_t* __restrict__ status_out,
           uint8_t* __restrict__ left_roi_out, const DprJob* __restrict__ jobs, int fuse_pyramid) {
  extern __shared__ __align__(16) uint8_t s_tile[];
  __shared__ DprShared S;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int64_t job = blockIdx.x / kCluster;
  const int crank = kCluster > 1 ? (int)(blockIdx.x % kCluster) : 0;     // == cluster.block_rank() for (kCluster,1,1) clusters
  const int64_t frame = job / n_hyp;
  if (mask != nullptr && mask[frame] == 0) return;     // skipped frame: none of its outputs is written (whole cluster)

  double* const Rc = S.Pc; double* const tc = S.Pc + 9;

  // ---- the plan of this refinement (dpr_prep_kernel), read by every thread so that staging starts at once --------
  const DprJob* jp = jobs + job;
  int4 ja, jb, jc;
  if (kCluster > 1 && jobs == nullptr) {
    // no setup launch: warp 0 builds the record in the (still unused) pyramid scratch; it is consumed before the first barrier
    // below, after which the scratch is free again
    DprJob* sj = reinterpret_cast<DprJob*>(s_tile + TILE_BYTES);
    if (wid == 0) dpr_prep_warp(pyr, cam, model, init + job * 6, sj, lane);
    __syncthreads();
    jp = sj;
    const int4* jw = reinterpret_cast<const int4*>(sj);
    ja = jw[0]; jb = jw[1]; jc = jw[2];
  } else {
    const int4* jw = reinterpret_cast<const int4*>(jp);
    ja = __ldg(jw); jb = __ldg(jw + 1); jc = __ldg(jw + 2);
  }
  const int lvl = ja.x;
  const bool build_level = fuse_pyramid != 0 && lvl > 0;
  auto stage_tile = [&]() {
    // stage the ROI tile with 16-byte asynchronous copies (LDGSTS): every chunk of a thread is in flight at once and
    // thread 0 sets up the LM state underneath them
    const int tx0 = jb.y, ty0 = jb.z, tw = jb.w, th = jc.x;
    const int lw = pyr.width[lvl];
    const int64_t lpitch = pyr.pitch[lvl];
    const uint8_t* limg = pyr.data[lvl] + frame * pyr.frame_stride[lvl];
    const uint8_t* src = limg + (int64_t)ty0 * lpitch + tx0;
    const bool vec = ((lpitch & 15) == 0) && ((reinterpret_cast<uintptr_t>(limg) & 15) == 0);
    const int chunks = tw > 0 ? (tw + 15) >> 4 : 1;
    const int rows = tw > 0 ? th : 0;                     // (an empty ROI stages nothing)
    const uint32_t sT0 = (uint32_t)__cvta_generic_to_shared(s_tile);
    int r = tid / chunks, c = tid - r * chunks;           // chunks <= 18: a step of 256 chunks is dr rows + dc columns
    const int dr = DPR_THREADS / chunks, dc = DPR_THREADS - dr * chunks;
    for (; r < rows; ) {
      const uint8_t* g = src + (int64_t)r * lpitch + 16 * c;
      if (vec && tx0 + 16 * c + 16 <= (int)lpitch) {
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" :: "r"(sT0 + r * TILE_PITCH + 16 * c), "l"(g) : "memory");
      } else {
        uint32_t w4[4] = {0, 0, 0, 0};
        for (int b = 0; b < 16; ++b)
          if (tx0 + 16 * c + b < lw) w4[b >> 2] |= (uint32_t)__ldcg(g + b) << (8 * (b & 3));
        *reinterpret_cast<uint4*>(s_tile + r * TILE_PITCH + 16 * c) = make_uint4(w4[0], w4[1], w4[2], w4[3]);
      }
      r += dr; c += dc;
      if (c >= chunks) { c -= chunks; ++r; }
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
  };
  if (!build_level) stage_tile();

  if (tid == 0) {
    S.cc = 0.0; S.lam = LAMBDA0; S.nc = 0; S.evals = 0; S.status = AGT_DPR_MAX_EVALS; S.alpha = 1.0; S.have_prev = 0;
    const double* p0 = init + job * 6;
    const DprJob* J = jp;
#pragma unroll
    for (int i = 0; i < 9; ++i) Rc[i] = J->R[i];
    tc[0] = p0[3]; tc[1] = p0[4]; tc[2] = p0[5];
    S.level = lvl;
    S.lw = pyr.width[lvl]; S.lh = pyr.height[lvl]; S.lpitch = pyr.pitch[lvl];
    S.limg = pyr.data[lvl] + frame * pyr.frame_stride[lvl];
    S.rx0 = ja.y; S.ry0 = ja.z; S.rx1 = ja.w; S.ry1 = jb.x;
    S.tx0 = jb.y; S.ty0 = jb.z; S.tw = jb.w; S.th = jc.x;
    S.left_roi = 0;
    double sc = 1.0 / (double)(1 << lvl);
    S.gscale = (float)(sc / 32.0);
    S.fx = (float)cam.fx; S.fy = (float)cam.fy;
    // active tags (visibility frozen at the initial pose)
    const uint32_t active = (uint32_t)jc.y;
    int na = 0, pre = 0;
    for (int k = 0; k < model.n_tags; ++k) {
      if (active >> k & 1u) {
        S.act_begin[na] = model.tag_begin[k];
        S.act_prefix[na] = pre;
        pre += model.tag_begin[k + 1] - model.tag_begin[k];
        ++na;
      }
    }
    S.act_prefix[na] = pre;
    S.n_active = na;
    S.proj[0] = cam.fx * sc; S.proj[1] = cam.fy * sc;
    S.proj[2] = cam.cx * sc; S.proj[3] = cam.cy * sc;
    S.projf[0] = (float)(cam.fx * sc); S.projf[1] = (float)(cam.fy * sc); S.projf[2] = (float)(cam.cx * sc); S.projf[3] = (float)(cam.cy * sc);
    S.zero = 0;
    publish_pose(S, Rc, tc);
    S.xbias = 0x41380000 + jb.y + 1; S.ybias = 0x41380000 + jb.z + 1;
    S.tw_m3 = jb.w >= 4 ? (uint32_t)(jb.w - 3) : 0u; S.th_m3 = jc.x >= 4 ? (uint32_t)(jc.x - 3) : 0u;
    S.stop = 0;
  }
  asm volatile("cp.async.wait_all;" ::: "memory");
  __syncthreads();
  if (build_level) {
    // K1 fused: only level 0 of the pyramid holds the frame.  Build the ROI of levels 1..l from it (intermediate levels
    // through the pyramid's own global buffers, which stay in L2), then stage the tile from the level just written.
    // Level 1 of an aligned frame (the usual case) is built by K1's own streaming warp routine, the eight warps
    // sharing the rows of the ROI; anything else by the generic band routine.
    uint8_t* s_scratch = s_tile + TILE_BYTES;
    bool tile_written = false;
    for (int L = 1; L <= lvl; ++L) {
      // rectangle needed at level L: the ROI at level l grown by the 5x5 support of every pyrDown above it
      int x0 = S.rx0, y0 = S.ry0, x1 = S.rx1, y1 = S.ry1;
      for (int m = lvl; m > L; --m) {
        x0 = max(0, 2 * x0 - 2) & ~15; y0 = max(0, 2 * y0 - 2);
        x1 = min(pyr.width[m - 1], 2 * ((x1 + 3) & ~3) + 2); y1 = min(pyr.height[m - 1], 2 * y1 + 2);
      }
      if (x1 > x0 && y1 > y0) {
        const uint8_t* simg = pyr.data[L - 1] + frame * pyr.frame_stride[L - 1];
        uint8_t* dimg = pyr.data[L] + frame * pyr.frame_stride[L];
        const int sw = pyr.width[L - 1], sh = pyr.height[L - 1], dw = pyr.width[L];
        const int64_t sp = pyr.pitch[L - 1], dp = pyr.pitch[L];
        // (only level 0 is read through the streaming routine: its 4-byte halo requests may be served by L1, which is
        // safe for data this launch never writes)
        const bool stream = L == 1 && (sw & 15) == 0 && sw >= 16 && sh >= 4 && (dw & 7) == 0 && (sp & 15) == 0 && (dp & 7) == 0 &&
                            (reinterpret_cast<uintptr_t>(simg) & 15) == 0 && (reinterpret_cast<uintptr_t>(dimg) & 7) == 0;
        if (stream) {
          constexpr int kQ = DPR_WARPS > 8 ? 2 : 3;                    // rows in flight per warp: 8 warps x 7 x 544 B of ring
          static_assert(DPR_WARPS * (kQ + 4) * 544 <= PB_BYTES, "ring of the streaming pyrDown");
          const uint32_t ring = (uint32_t)__cvta_generic_to_shared(s_scratch) + wid * ((kQ + 4) * 544);
          const int xo1 = min(dw, (x1 + 7) & ~7);
          const int per = (y1 - y0 + DPR_WARPS - 1) / DPR_WARPS;
          const int oy0 = y0 + wid * per, oy1 = min(oy0 + per, y1);
          if (oy0 < oy1)
            for (int xb = x0; xb < xo1; xb += 256)
              agt_pyr_down_strip<kQ, 1>(simg, sw, sh, sp, dimg, dp, xb + 8 * lane, xo1, oy0, oy1, lane, ring);
          asm volatile("cp.async.wait_all;" ::: "memory");
        } else {
          uint8_t* s_in = s_scratch;
          uint16_t* s_h = reinterpret_cast<uint16_t*>(s_in + 2 * PB_IN_ROWS * PB_IN_PITCH);
          cta_pyr_down_region(simg, sw, sh, sp, dimg, dp, L == lvl ? s_tile : nullptr, S.tx0, S.ty0, S.tw, S.th, x0, y0, x1, y1, s_in, s_h);
          tile_written = tile_written || L == lvl;
        }
      }
      __syncthreads();
    }
    if (!tile_written) {                                              // (uniform across the CTA)
      stage_tile();
      asm volatile("cp.async.wait_all;" ::: "memory");
      __syncthreads();
    }
  }

  const int n_act_samples = S.act_prefix[S.n_active];
  const float fx = S.fx, fy = S.fy, gsc = S.gscale;
  const int lw = S.lw, lh = S.lh, tx0 = S.tx0, ty0 = S.ty0;
  const int64_t lpitch = S.lpitch;
  const uint8_t* limg = S.limg;
  // footprint origin relative to the tile straight from the high word of ul + 1.5 * 2^20 (see the sample loop)
  const int xbias = S.xbias, ybias = S.ybias;
  const int xoff = tx0 + 1, yoff = ty0 + 1;
  const f32x2 fl2 = pk2(S.projf[0], S.projf[1]), cl2 = pk2(S.projf[2], S.projf[3]);
  const uint32_t tw_m3 = S.tw_m3, th_m3 = S.th_m3;
  const f32x2 fg = pk2(fx * gsc, fy * gsc);
  const uint32_t sP = smem_addr(S.Rd), sT = smem_addr(s_tile);
  // dp4a coefficient words from constant memory: they stay in uniform registers across the loop
  const int cDX0_3 = kCoef[0], cDX0_10 = kCoef[1], cDX1_3 = kCoef[2], cDX1_10 = kCoef[3], cSM0 = kCoef[4], cSM1 = kCoef[5],
            cSM0_NEG = kCoef[6], cSM1_NEG = kCoef[7];

  for (int it = 0;; ++it) {
    // ================= evaluate cost + normal equations at the trial pose =================
    // Internal order of the six Jacobian columns: q = (J0, -J1, J3, J4, J2, J5) in three pairs QA QB QC, chosen so that
    // every pair is produced as a pair (no register moves); signs and order are undone when the sums are unpacked.
    f32x2 p0 = 0, p1 = 0, p2 = 0, p3 = 0, p4 = 0, p5 = 0, p6 = 0, p7 = 0, p8 = 0, p9 = 0, p10 = 0, p11 = 0;
    float s11 = 0.f, s44 = 0.f, s55 = 0.f, scost = 0.f;
    int cnt = 0;
    // rotation / translation of the trial pose: float64 copy (shared memory) for the projection, float32 for the Jacobian
    const f32x2* Rp = reinterpret_cast<const f32x2*>(S.Rf);
    const f32x2 R03 = Rp[0], R14 = Rp[1], R25 = Rp[2], t01 = Rp[3];
    const float R6 = S.Rf[8], R7 = S.Rf[9], R8 = S.Rf[10], t2 = S.Rf[11];
    // One sample: projection, footprint fetch, Scharr taps, residual, Jacobian, normal-equation products.
    auto eval_sample = [&](const float4 sm) {
      // float32 lever arm Y = R x for the Jacobian and the reciprocal-depth seed (rounding of these only perturbs
      // the LM step, not the cost)
      const f32x2 Yxy = fma2(R25, bc2(sm.z), fma2(R14, bc2(sm.y), mul2(R03, bc2(sm.x))));
      const float Yz = fmaf(R8, sm.z, fmaf(R7, sm.y, R6 * sm.x));
      const float Z32 = Yz + t2;
      float iz;
      asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(iz) : "f"(Z32));             // MUFU.RCP: Jacobian + Newton seed
#if AGT_DPR_F32_PROJECTION
      // Projection in float32.  Round 1 needed float64 here: its LM accepted a step only if the cost went down, near convergence
      // that compares costs 1e-6 apart, and float32 pixel coordinates (ulp 1e-4 px at 1080p) flipped 20 % of those decisions.
      // The loop now accepts within a 1e-2 slack and contracts onto J^T r = 0 (oracle/dpr_oracle.py), so that noise only moves
      // the fixed point by ~1e-8 rad, and the projection is the camera-frame (X, Y) the Jacobian needs anyway times a Newton-
      // refined reciprocal depth: 11 instructions instead of 28 (13 of them DFMA at two issue cycles each).
      const float iz1 = iz * fmaf(-Z32, iz, 2.f);
      const f32x2 XY = add2(Yxy, t01);
      const f32x2 uv = fma2(mul2(XY, fl2), bc2(iz1), cl2);                 // (ul, vl)
      const float fu = floorf(lo2(uv)), fv = floorf(hi2(uv));
      const int lx = __float2int_rd(lo2(uv)) - xoff, ly = __float2int_rd(hi2(uv)) - yoff;   // footprint origin in the tile
      const bool depth_ok = Z32 > 1e-6f;
#else
      // Projection in float64: the accept/reject decisions of the LM loop compare costs that differ by ~1e-6
      // relative near convergence; float32 pixel coordinates (ulp 6e-5 px at 1080p) add ~1e-6 of noise to the
      // cost and flip 20 % of those decisions, float64 leaves 0.2 % (profiles/r01_dpr_precision_sweep.log).
      const double sx = sm.x, sy = sm.y, sz = sm.z;
      // (the float64 pose is read from shared memory with broadcast loads: 24 registers less per thread)
      const double2 p01 = lds_f64x2(sP), p23 = lds_f64x2(sP + 16), p45 = lds_f64x2(sP + 32), p67 = lds_f64x2(sP + 48),
                    p8t = lds_f64x2(sP + 64), ptt = lds_f64x2(sP + 80);
      // homogeneous level-l pixel coordinates (K_l folded into the pose by the LM thread): (ul dZ, vl dZ, dZ)
      const double dX = fma(p01.x, sx, fma(p01.y, sy, fma(p23.x, sz, p8t.y)));
      const double dY = fma(p23.y, sx, fma(p45.x, sy, fma(p45.y, sz, ptt.x)));
      const double dZ = fma(p67.x, sx, fma(p67.y, sy, fma(p8t.x, sz, ptt.y)));
      double r0 = (double)iz;                         // 2^-22 relative; one Newton step -> 2^-44 (4e-11 px at 1080p)
      r0 = r0 * (2.0 - dZ * r0);
      // floor + fraction without conversions or float64 compares: ul + 1.5 * 2^20 (one FMA rounding down) leaves
      // floor(ul) in the low bits of the high mantissa word and the fraction, scaled by 2^32, in the low word;
      // NaN / Inf / |ul| >= 2^19 give a high word far outside any image
      const double kMagic = 1572864.0;
      const double tu = __fma_rd(dX, r0, kMagic), tv = __fma_rd(dY, r0, kMagic);
      const int lx = __double2hiint(tu) - xbias, ly = __double2hiint(tv) - ybias;     // footprint origin in the tile
      const bool depth_ok = dZ > 1e-6;
#endif
      // 4x4 footprint rows y0-1..y0+2, columns x0-1..x0+2
      uint32_t row[4];
      if (Z32 > 2e-6f && (uint32_t)lx < tw_m3 && (uint32_t)ly < th_m3) {
        // (float32 depth above 2e-6 implies float64 depth above 1e-6; the tile lies inside the level image, so a
        // footprint inside the tile is a valid sample)
        const uint32_t a0 = sT + ly * TILE_PITCH + (lx & ~3);
        const uint32_t sel = 0x3210 + 0x1111 * (lx & 3);
#pragma unroll
        for (int r = 0; r < 4; ++r) row[r] = __byte_perm(lds_u32(a0 + r * TILE_PITCH), lds_u32(a0 + r * TILE_PITCH + 4), sel);
      } else {
        const int x0 = lx + tx0 + 1, y0 = ly + ty0 + 1;
        // valid <=> z > 1e-6 and 1 <= floor(ul) <= lw-3 and 1 <= floor(vl) <= lh-3
        if (!depth_ok || x0 < 1 || x0 > lw - 3 || y0 < 1 || y0 > lh - 3) return;
        if (x0 - 1 < S.rx0 || y0 - 1 < S.ry0 || x0 + 3 > S.rx1 || y0 + 3 > S.ry1) S.left_roi = 1;   // benign race: all write 1
        const uint8_t* g = limg + (int64_t)(y0 - 1) * lpitch + (x0 - 1);
#pragma unroll
        for (int r = 0; r < 4; ++r) row[r] = ld4_global(g + r * lpitch);
      }
      // bilinear weights; (a, b) = fractions of (ul, vl)
#if AGT_DPR_F32_PROJECTION
      const f32x2 ab = add2(uv, pk2(-fu, -fv));
#else
      const f32x2 ab = mul2(pk2((float)(uint32_t)__double2loint(tu), (float)(uint32_t)__double2loint(tv)), bc2(2.3283064365386963e-10f));
#endif
      const f32x2 omab = fma2(ab, bc2(-1.f), bc2(1.f));                     // (1-a, 1-b)
      const f32x2 wx = mul2(ab, swap2(omab));                               // (w01, w10) = (a (1-b), b (1-a))
      const float w00 = lo2(omab) * hi2(omab), w11 = lo2(ab) * hi2(ab), w01 = lo2(wx), w10 = hi2(wx);
      // Scharr at (x0,y0) (x0+1,y0) (x0,y0+1) (x0+1,y0+1): the [3 10 3] row weights are folded into the byte
      // coefficients and the three rows are chained through the dp4a accumulator, which starts at the bit pattern of
      // 1.5 * 2^23: the integer sum lands in the mantissa and one packed subtraction turns two taps into floats
      const int kB = 0x4B400000;
      const f32x2 kNegBias = bc2(-12582912.f);
      const f32x2 g00 = add2(pk2(dp4c(row[2], cDX0_3, dp4c(row[1], cDX0_10, dp4c(row[0], cDX0_3, kB))),
                                 dp4c(row[2], cSM0, dp4c(row[0], cSM0_NEG, kB))), kNegBias);
      const f32x2 g01 = add2(pk2(dp4c(row[2], cDX1_3, dp4c(row[1], cDX1_10, dp4c(row[0], cDX1_3, kB))),
                                 dp4c(row[2], cSM1, dp4c(row[0], cSM1_NEG, kB))), kNegBias);
      const f32x2 g10 = add2(pk2(dp4c(row[3], cDX0_3, dp4c(row[2], cDX0_10, dp4c(row[1], cDX0_3, kB))),
                                 dp4c(row[3], cSM0, dp4c(row[1], cSM0_NEG, kB))), kNegBias);
      const f32x2 g11 = add2(pk2(dp4c(row[3], cDX1_3, dp4c(row[2], cDX1_10, dp4c(row[1], cDX1_3, kB))),
                                 dp4c(row[3], cSM1, dp4c(row[1], cSM1_NEG, kB))), kNegBias);
      const float i00 = (float)((row[1] >> 8) & 0xffu), i01 = (float)((row[1] >> 16) & 0xffu);
      const float i10 = (float)((row[2] >> 8) & 0xffu), i11 = (float)((row[2] >> 16) & 0xffu);
      const float I = w00 * i00 + w01 * i01 + w10 * i10 + w11 * i11;
      const f32x2 G = fma2(bc2(w11), g11, fma2(bc2(w10), g10, fma2(bc2(w01), g01, mul2(bc2(w00), g00))));   // (Gx, Gy) * 32 * 2^l
      const float r = I - sm.w;
      const f32x2 QB = mul2(mul2(G, fg), bc2(iz));                          // (g0, g1) = (J3, J4)
#if !AGT_DPR_F32_PROJECTION
      const f32x2 XY = add2(Yxy, t01);
#endif
      const float g0 = lo2(QB), g1 = hi2(QB);
      const float g2 = -(g0 * lo2(XY) + g1 * hi2(XY)) * iz;
      // (J0, -J1) = g2 (Yy, Yx) - Yz (g1, g0);  J2 = Yx g1 - Yy g0
      const f32x2 QA = fma2(bc2(g2), swap2(Yxy), mul2(bc2(-Yz), swap2(QB)));
      const f32x2 QC = pk2(lo2(Yxy) * g1 - hi2(Yxy) * g0, g2);             // (J2, J5)
      const float q0 = lo2(QA), q1 = hi2(QA), q4 = lo2(QC);
      p0 = fma2(bc2(q0), QA, p0); p1 = fma2(bc2(q0), QB, p1); p2 = fma2(bc2(q0), QC, p2);
      p3 = fma2(bc2(q1), QB, p3); p4 = fma2(bc2(q1), QC, p4);
      p5 = fma2(bc2(g0), QB, p5); p6 = fma2(bc2(g0), QC, p6);
      p7 = fma2(bc2(g1), QC, p7); p8 = fma2(bc2(q4), QC, p8);
      p9 = fma2(bc2(r), QA, p9); p10 = fma2(bc2(r), QB, p10); p11 = fma2(bc2(r), QC, p11);
      s11 = fmaf(q1, q1, s11); s44 = fmaf(g1, g1, s44); s55 = fmaf(g2, g2, s55);
      // the per-thread cost (<= ~30 terms) in float32: its rounding (1e-8 relative) is below that of the
      // float32 interpolation feeding it; across threads it is summed in float64
      scost = fmaf(r, r, scost);
      ++cnt;
    };
    // This thread's samples are j0, j0 + step, ... of the concatenated active tags.  Software pipeline: the model
    // record of the next sample is requested before the current one is consumed; two copies of the body alternate
    // between two record registers so that nothing has to be moved.
    const int step = kCluster * DPR_THREADS;
    const int j0 = crank * DPR_THREADS + tid;
    int left = j0 < n_act_samples ? (n_act_samples - j0 + step - 1) / step : 0;
    if (left > 0) {
      int seg = 0;
      while (j0 >= S.act_prefix[seg + 1]) ++seg;
      int sidx = S.act_begin[seg] + (j0 - S.act_prefix[seg]);               // record index of the current sample
      int seg_last = S.act_begin[seg] + (S.act_prefix[seg + 1] - S.act_prefix[seg]);   // end of this tag's records
      auto advance = [&]() {
        sidx += step;
        if (sidx >= seg_last) {                        // crossed into the next active tag (rare)
          int j = S.act_prefix[seg + 1] + (sidx - seg_last);
          do { ++seg; } while (j >= S.act_prefix[seg + 1]);
          sidx = S.act_begin[seg] + (j - S.act_prefix[seg]);
          seg_last = S.act_begin[seg] + (S.act_prefix[seg + 1] - S.act_prefix[seg]);
        }
      };
      // The address of each request is made to depend on the record about to be consumed: the scoreboards count
      // outstanding loads, so a request issued just before the first use of the previous record would make that use
      // wait for the new request as well (seen as 11 % of all stall samples on one instruction).
      const int zero = S.zero;
      float4 smA = __ldg(&samples[sidx]), smB;
#pragma unroll 1
      while (true) {
        const bool moreA = left > 1;
        if (moreA) advance();
        smB = __ldg(&samples[sidx + (__float_as_int(smA.w) & zero)]);     // (the last sample re-reads its own record)
        eval_sample(smA);
        if (!moreA) break;
        const bool moreB = left > 2;
        if (moreB) advance();
        smA = __ldg(&samples[sidx + (__float_as_int(smB.w) & zero)]);
        eval_sample(smB);
        if (!moreB) break;
        left -= 2;
      }
    }
    // ---- reduce: one transposing butterfly over the 27 sums, float64 across warps --------------------
    // After the step with offset h a lane keeps the half of the values whose index has bit h equal to its own lane
    // bit, so 31 shuffles (instead of 27 x 5) leave the total of sum k on lane k - the same summation tree as a
    // butterfly all-reduce.
    {
      float v[32];
      v[0] = lo2(p0);   v[1] = -hi2(p0);  v[2] = lo2(p2);   v[3] = lo2(p1);   v[4] = hi2(p1);   v[5] = hi2(p2);
      v[6] = s11;       v[7] = -lo2(p4);  v[8] = -lo2(p3);  v[9] = -hi2(p3);  v[10] = -hi2(p4);
      v[11] = lo2(p8);  v[12] = lo2(p6);  v[13] = lo2(p7);  v[14] = hi2(p8);
      v[15] = lo2(p5);  v[16] = hi2(p5);  v[17] = hi2(p6);  v[18] = s44;      v[19] = hi2(p7);  v[20] = s55;
      v[21] = lo2(p9);  v[22] = -hi2(p9); v[23] = lo2(p11); v[24] = lo2(p10); v[25] = hi2(p10); v[26] = hi2(p11);
#pragma unroll
      for (int k = 27; k < 32; ++k) v[k] = 0.f;
#pragma unroll
      for (int h = 16; h >= 1; h >>= 1) {
        const bool up = (lane & h) != 0;
#pragma unroll
        for (int k = 0; k < h; ++k) {
          const float keep = up ? v[k + h] : v[k], send = up ? v[k] : v[k + h];
          v[k] = keep + __shfl_xor_sync(0xffffffffu, send, h);
        }
      }
      const double cost = agt_warp_sum((double)scost);
      cnt = __reduce_add_sync(0xffffffffu, cnt);
      double o = (double)v[0];
      if (lane == 27) o = cost;
      if (lane == 28) o = (double)cnt;
      if (lane < 29) S.wsum[wid][lane] = o;
    }
    __syncthreads();
    double tot = 0.0;                                     // lane k of warp 0: sum k over the CTA (then the cluster)
    if (wid == 0 && lane < 29) {
#pragma unroll
      for (int w = 0; w < DPR_WARPS; ++w) tot += S.wsum[w][lane];
    }
    if (kCluster > 1) {
      // Every CTA of the cluster adds up every CTA's partial sums, in rank order, and then takes the LM step itself: the
      // same numbers through the same operations, so all of them arrive at the same decision and the same next pose, and
      // one cluster barrier per evaluation is enough (nobody waits for CTA 0 to publish the pose).  The exchange buffer is
      // double-buffered by evaluation parity: a CTA overwrites a buffer only after the barrier of the next evaluation,
      // which every CTA reaches after it has read this one.
      cg::cluster_group cluster = cg::this_cluster();
      if (wid == 0 && lane < 29) S.tot[it & 1][lane] = tot;
      cluster.sync();                                   // every CTA's partial sums are in its S.tot
      if (wid == 0 && lane < 29) {
        tot = 0.0;
        for (int r = 0; r < kCluster; ++r) tot += cluster.map_shared_rank(&S, r)->tot[it & 1][lane];
      }
    }

    // ================= LM bookkeeping (warp 0: decisions in every lane, the 6x6 solve in lane 0) ==========
    if (wid == 0) {
      const double cn = 0.5 * __shfl_sync(0xffffffffu, tot, 27);
      const int nn = (int)__shfl_sync(0xffffffffu, tot, 28);
      double cc = S.cc, lam = S.lam;
      const int evals = S.evals + 1;
      int status = S.status;
      bool need_step = false, accept = false;
      if (evals == 1) {
        accept = true;
        if (nn == 0) status = AGT_DPR_NONE; else need_step = true;
      } else {
        // |step| against the tolerances, squared on both sides (no square root on the critical path)
        const double* ds = S.dstep;
        const double nw2 = ds[0] * ds[0] + ds[1] * ds[1] + ds[2] * ds[2], nt2 = ds[3] * ds[3] + ds[4] * ds[4] + ds[5] * ds[5];
        if (nn > 0 && cn < cc * (1.0 + ACCEPT_SLACK) && cn <= S.c0) {
          accept = true;
          lam = fmax(lam * 0.1, LAMBDA_MIN);
          if (nw2 < TOL_ROT * TOL_ROT && nt2 < TOL_TRANS * TOL_TRANS) status = AGT_DPR_CONVERGED; else need_step = true;
        } else {
          lam *= 10.0;
          if (nw2 < TOL_ROT * TOL_ROT && nt2 < TOL_TRANS * TOL_TRANS) status = AGT_DPR_CONVERGED;
          else if (lam > LAMBDA_MAX) status = AGT_DPR_LAMBDA;
          else need_step = true;
        }
      }
      if (accept) {                                       // the trial pose and its normal equations become current
        if (lane < 27) S.Hb[lane] = tot;
        if (lane < 12) S.Pc[lane] = S.Pt[lane];
        cc = cn;
      }
      if (need_step && evals >= MAX_EVALS) need_step = false;     // status stays MAX_EVALS
      __syncwarp();
      if (lane == 0) {
        double alpha = S.alpha;
        int have_prev = S.have_prev;
        if (evals > 1) {
          if (accept) {
#pragma unroll
            for (int q = 0; q < 6; ++q) S.dprev[q] = S.dgn[q];
            have_prev = S.lam <= LAMBDA0;        // S.lam: the damping the accepted step was solved with
          } else {
            have_prev = 0;
            alpha = 1.0;
          }
        }
        while (need_step) {
          double A[21], d[6];
#pragma unroll
          for (int k = 0; k < 21; ++k) A[k] = S.Hb[k];
#pragma unroll
          for (int q = 0; q < 6; ++q) { A[agt_hk(q, q)] = fma(lam, A[agt_hk(q, q)], A[agt_hk(q, q)]); d[q] = -S.Hb[21 + q]; }
          if (agt_chol6_packed(A, d)) {
            if (lam > LAMBDA0) {             // damped steps are not comparable: no step-length adaptation
              alpha = 1.0;
              have_prev = 0;
            } else if (have_prev) {
              // ratio of this step to the previous accepted one, in the metric of the current H
              double num = 0.0, den = 0.0, dd = 0.0;
#pragma unroll
              for (int q = 0; q < 6; ++q) {
                double a = 0.0, b = 0.0;
#pragma unroll
                for (int r = 0; r < 6; ++r) {
                  const double h = S.Hb[q <= r ? agt_hk(q, r) : agt_hk(r, q)];
                  a = fma(h, S.dprev[r], a);
                  b = fma(h, d[r], b);
                }
                num = fma(d[q], a, num); den = fma(S.dprev[q], a, den); dd = fma(d[q], b, dd);
              }
              if (num * num > AITKEN_COS2 * den * dd) alpha = fmin(fmax(alpha / (1.0 - fmin(num / den, AITKEN_QMAX)), ALPHA_MIN), ALPHA_MAX);
              else alpha = 1.0 + 0.5 * (alpha - 1.0);
            }
#pragma unroll
            for (int q = 0; q < 6; ++q) { S.dgn[q] = d[q]; d[q] *= alpha; S.dstep[q] = d[q]; }
            double E[9], Rt[9], tt[3];
            rodrigues_step(d, E);
#pragma unroll
            for (int r = 0; r < 3; ++r)
#pragma unroll
              for (int c = 0; c < 3; ++c) Rt[r * 3 + c] = E[r * 3] * Rc[c] + E[r * 3 + 1] * Rc[3 + c] + E[r * 3 + 2] * Rc[6 + c];
#pragma unroll
            for (int q = 0; q < 3; ++q) tt[q] = tc[q] + d[3 + q];
            publish_pose(S, Rt, tt);
            break;
          }
          lam *= 10.0;
          if (lam > LAMBDA_MAX) { status = AGT_DPR_LAMBDA; need_step = false; }
        }
        S.alpha = alpha; S.have_prev = have_prev;
        S.stop = need_step ? 0 : 1;
        S.cc = cc; S.lam = lam; S.evals = evals; S.status = status;
        if (evals == 1) S.c0 = cn;
        if (accept) S.nc = nn;
      }
    }
    __syncthreads();
    if (S.stop) break;
  }
  if (kCluster > 1) {
    cg::cluster_group cluster = cg::this_cluster();
    cluster.sync();
    if (crank == 0 && tid == 0)
      for (int r = 1; r < kCluster; ++r) S.left_roi |= cluster.map_shared_rank(&S, r)->left_roi;
    cluster.sync();                                     // keep every CTA's shared memory alive until CTA 0 has read it
    if (crank != 0) return;
  }

  if (tid == 0) {
    double rv[3];
    agt_log_rotation(Rc, rv);
    double* po = pose_out + job * 6;
    po[0] = rv[0]; po[1] = rv[1]; po[2] = rv[2]; po[3] = tc[0]; po[4] = tc[1]; po[5] = tc[2];
    if (cost_out) cost_out[job] = (float)S.cc;
    if (nvalid_out) nvalid_out[job] = S.nc;
    if (evals_out) evals_out[job] = S.evals;
    if (status_out) status_out[job] = (uint8_t)S.status;
    if (left_roi_out) left_roi_out[job] = (uint8_t)S.left_roi;
  }
}

__global__ void dpr_rects_kernel(agt_pyramid pyr, agt_camera cam, double pitch, double radius, const double* __restrict__ init,
                                 int n_hyp, int32_t* __restrict__ rects, int batch) {
  int f = blockIdx.x * blockDim.x + threadIdx.x;
  if (f >= batch) return;
  int32_t r[4];
  agt_dpr_rect_l0(cam, pitch, radius, init + (int64_t)f * n_hyp * 6, n_hyp, pyr.width, pyr.height, pyr.levels, r);
  *reinterpret_cast<int4*>(rects + (int64_t)f * 4) = make_int4(r[0], r[1], r[2], r[3]);
}

__global__ void any_flag_kernel(const uint8_t* __restrict__ flags, int stride, uint8_t* __restrict__ out, int batch) {
  int f = blockIdx.x * blockDim.x + threadIdx.x;
  if (f >= batch) return;
  uint8_t any = 0;
  for (int k = 0; k < stride; ++k) any |= flags[(int64_t)f * stride + k];
  out[f] = any ? 1 : 0;
}

__global__ void select_best_kernel(const double* __restrict__ pose, const float* __restrict__ cost,
                                   const int32_t* __restrict__ nvalid, int n_hyp, int32_t* __restrict__ best,
                                   double* __restrict__ best_pose, int batch) {
  // one warp per frame: lowest index among the hypotheses whose score 2c/n is within SELECT_TIE of the minimum.  Runs that end
  // in the same fixed point have scores that agree to ~1e-6 (their last steps, float32 sums); comparing them exactly would
  // make the winning INDEX depend on that noise, so everything within 1e-4 of the best counts as a tie -> lowest index.
  constexpr double SELECT_TIE = 1e-4;
  int f = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  int lane = threadIdx.x & 31;
  if (f >= batch) return;
  double bs = INFINITY;
  for (int h = lane; h < n_hyp; h += 32) {
    int n = nvalid[(int64_t)f * n_hyp + h];
    double s = n > 0 ? 2.0 * (double)cost[(int64_t)f * n_hyp + h] / (double)n : INFINITY;
    bs = fmin(bs, s);
  }
  for (int o = 16; o > 0; o >>= 1) bs = fmin(bs, __shfl_xor_sync(0xffffffffu, bs, o));
  const double limit = bs * (1.0 + SELECT_TIE);
  int bi = 0x7fffffff;
  for (int h = lane; h < n_hyp; h += 32) {
    int n = nvalid[(int64_t)f * n_hyp + h];
    double s = n > 0 ? 2.0 * (double)cost[(int64_t)f * n_hyp + h] / (double)n : INFINITY;
    if (s <= limit && s < INFINITY && h < bi) bi = h;
  }
  for (int o = 16; o > 0; o >>= 1) bi = min(bi, __shfl_xor_sync(0xffffffffu, bi, o));
  if (bi == 0x7fffffff) bi = 0;
  if (lane == 0) best[f] = bi;
  if (best_pose && lane < 6) best_pose[(int64_t)f * 6 + lane] = pose[((int64_t)f * n_hyp + bi) * 6 + lane];
}

}  // namespace

static int refine_impl(agt_ctx* ctx, const agt_pyramid* pyr, const double* d_init, int n_hyp, const uint8_t* d_mask,
                       double* d_pose, float* d_cost, int32_t* d_n_valid, int32_t* d_evals, uint8_t* d_status,
                       uint8_t* d_left_roi, int batch, int fuse_pyramid) {
  if (!ctx) return AGT_ERR_INVALID;
  if (batch == 0) return AGT_OK;          // nothing to do (empty tensors may carry null pointers)
  if (!ctx->camera_set || !ctx->model_set) AGT_FAIL(ctx, AGT_ERR_NOT_READY, "agt_refine: camera and surface model must be set");
  if (!pyr || !d_init || !d_pose || n_hyp < 1 || batch < 0) AGT_FAIL(ctx, AGT_ERR_INVALID, "agt_refine: bad arguments");
  if (pyr->levels < 1 || pyr->levels > AGT_MAX_LEVELS) AGT_FAIL(ctx, AGT_ERR_INVALID, "agt_refine: bad pyramid descriptor");
  if (ctx->cam.has_dist) AGT_FAIL(ctx, AGT_ERR_INVALID, "agt_refine: lens distortion is not supported; undistort the frame first (detect_pose.py:611-619)");
  int64_t jobs = (int64_t)batch * n_hyp;
  if (jobs == 0) return AGT_OK;
  if (jobs > 0x7fffffffLL) AGT_FAIL(ctx, AGT_ERR_INVALID, "agt_refine: batch*n_hyp too large");
  static bool attr_set[64] = {false};
  if (!attr_set[ctx->device & 63]) {
    AGT_CUDA(ctx, cudaFuncSetAttribute(dpr_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, TILE_BYTES + PB_BYTES));
    AGT_CUDA(ctx, cudaFuncSetAttribute(dpr_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, TILE_BYTES + PB_BYTES));
    AGT_CUDA(ctx, cudaFuncSetAttribute(dpr_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, TILE_BYTES + PB_BYTES));
    AGT_CUDA(ctx, cudaFuncSetAttribute(dpr_kernel<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, TILE_BYTES + PB_BYTES));
    attr_set[ctx->device & 63] = true;
  }
  // 2 CTAs/SM at 128 registers: a 3-CTA build (80 registers) spills in the sample loop and measured 20 % slower.
  // Small batches (fewer refinements than 2 CTA slots per SM) are spread over clusters of 2 / 4 / 8 CTAs.
  DprJob* d_jobs = nullptr;
  {
    void* pj = nullptr;
    int rc = agt_scratch(ctx, 5, sizeof(DprJob) * (size_t)jobs, &pj);
    if (rc) return rc;
    d_jobs = static_cast<DprJob*>(pj);
  }
  int cluster = 1;
  const int64_t slots = 2LL * ctx->sm_count;
  while (cluster < 8 && jobs * (cluster * 2) <= slots) cluster *= 2;
  if (cluster == 1) {
    dpr_prep_kernel<<<(unsigned)((jobs + 127) / 128), 128, 0, ctx->stream>>>(*pyr, ctx->cam, ctx->model, d_init, n_hyp, d_mask, d_jobs, jobs);
    AGT_LAUNCH_CHECK(ctx);
  } else {
    d_jobs = nullptr;                    // cluster launches derive the setup record in the kernel (dpr_prep_warp)
  }
  if (cluster == 1) {
    dpr_kernel<1><<<(unsigned)jobs, DPR_THREADS, TILE_BYTES + PB_BYTES, ctx->stream>>>(*pyr, ctx->cam, ctx->model.samples, ctx->model, d_init,
                                                                         n_hyp, d_mask, d_pose, d_cost, d_n_valid, d_evals, d_status,
                                                                         d_left_roi, d_jobs, fuse_pyramid);
  } else {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)(jobs * cluster));
    cfg.blockDim = dim3(DPR_THREADS);
    cfg.dynamicSmemBytes = TILE_BYTES + PB_BYTES;
    cfg.stream = ctx->stream;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = cluster; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    agt_pyramid pv = *pyr;
    const float4* smp = ctx->model.samples;
    cudaError_t e;
    if (cluster == 2)
      e = cudaLaunchKernelEx(&cfg, dpr_kernel<2>, pv, ctx->cam, smp, ctx->model, d_init, n_hyp, d_mask, d_pose, d_cost, d_n_valid, d_evals, d_status, d_left_roi, (const DprJob*)d_jobs, fuse_pyramid);
    else if (cluster == 4)
      e = cudaLaunchKernelEx(&cfg, dpr_kernel<4>, pv, ctx->cam, smp, ctx->model, d_init, n_hyp, d_mask, d_pose, d_cost, d_n_valid, d_evals, d_status, d_left_roi, (const DprJob*)d_jobs, fuse_pyramid);
    else
      e = cudaLaunchKernelEx(&cfg, dpr_kernel<8>, pv, ctx->cam, smp, ctx->model, d_init, n_hyp, d_mask, d_pose, d_cost, d_n_valid, d_evals, d_status, d_left_roi, (const DprJob*)d_jobs, fuse_pyramid);
    if (e != cudaSuccess) AGT_FAIL(ctx, AGT_ERR_CUDA, "agt_refine: cluster launch failed: %s", cudaGetErrorString(e));
  }
  AGT_LAUNCH_CHECK(ctx);
  return AGT_OK;
}

extern "C" int agt_refine(agt_ctx* ctx, const agt_pyramid* pyr, const double* d_init, int n_hyp, const uint8_t* d_mask,
                          double* d_pose, float* d_cost, int32_t* d_n_valid, int32_t* d_evals, uint8_t* d_status,
                          uint8_t* d_left_roi, int batch) {
  return refine_impl(ctx, pyr, d_init, n_hyp, d_mask, d_pose, d_cost, d_n_valid, d_evals, d_status, d_left_roi, batch, 0);
}

extern "C" int agt_refine_fused(agt_ctx* ctx, const agt_pyramid* pyr, const double* d_init, int n_hyp, const uint8_t* d_mask,
                                double* d_pose, float* d_cost, int32_t* d_n_valid, int32_t* d_evals, uint8_t* d_status,
                                uint8_t* d_left_roi, int batch) {
  return refine_impl(ctx, pyr, d_init, n_hyp, d_mask, d_pose, d_cost, d_n_valid, d_evals, d_status, d_left_roi, batch, 1);
}

extern "C" int agt_select_best(agt_ctx* ctx, const double* d_pose, const float* d_cost, const int32_t* d_n_valid,
                               int n_hyp, int32_t* d_best, double* d_best_pose, int batch) {
  if (!ctx) return AGT_ERR_INVALID;
  if (batch == 0) return AGT_OK;          // nothing to do (empty tensors may carry null pointers)
  if (!d_pose || !d_cost || !d_n_valid || !d_best || n_hyp < 1 || batch < 0)
    AGT_FAIL(ctx, AGT_ERR_INVALID, "agt_select_best: bad arguments");
  if (batch == 0) return AGT_OK;
  int threads = 128;
  int blocks = (int)(((int64_t)batch * 32 + threads - 1) / threads);
  select_best_kernel<<<blocks, threads, 0, ctx->stream>>>(d_pose, d_cost, d_n_valid, n_hyp, d_best, d_best_pose, batch);
  AGT_LAUNCH_CHECK(ctx);
  return AGT_OK;
}

extern "C" int agt_dpr_rects(agt_ctx* ctx, const agt_pyramid* pyr, const double* d_init, int n_hyp, int32_t* d_rects, int batch) {
  if (!ctx) return AGT_ERR_INVALID;
  if (batch == 0) return AGT_OK;          // nothing to do (empty tensors may carry null pointers)
  if (!ctx->camera_set || !ctx->model_set) AGT_FAIL(ctx, AGT_ERR_NOT_READY, "agt_dpr_rects: camera and surface model must be set");
  if (!pyr || !d_init || !d_rects || n_hyp < 1 || batch < 0 || (reinterpret_cast<uintptr_t>(d_rects) & 15))
    AGT_FAIL(ctx, AGT_ERR_INVALID, "agt_dpr_rects: bad arguments (d_rects must be 16-byte aligned)");
  if (batch == 0) return AGT_OK;
  dpr_rects_kernel<<<(batch + 127) / 128, 128, 0, ctx->stream>>>(*pyr, ctx->cam, ctx->model.pitch, ctx->model.radius, d_init, n_hyp,
                                                                d_rects, batch);
  AGT_LAUNCH_CHECK(ctx);
  return AGT_OK;
}

extern "C" int agt_any_flag(agt_ctx* ctx, const uint8_t* d_flags, int stride, uint8_t* d_out, int batch) {
  if (!ctx) return AGT_ERR_INVALID;
  if (batch == 0) return AGT_OK;          // nothing to do (empty tensors may carry null pointers)
  if (!d_flags || !d_out || stride < 1 || batch < 0) AGT_FAIL(ctx, AGT_ERR_INVALID, "agt_any_flag: bad arguments");
  if (batch == 0) return AGT_OK;
  any_flag_kernel<<<(batch + 127) / 128, 128, 0, ctx->stream>>>(d_flags, stride, d_out, batch);
  AGT_LAUNCH_CHECK(ctx);
  return AGT_OK;
}
