// Streaming cv::pyrDown of one strip of output rows by one warp: the core of K1 (agt_pyramid.cu) and of the K1 stage
// fused into the dense-refinement kernel (agt_dpr.cu).  See the comments in agt_pyramid.cu for the design.
#pragma once
#include "agt_common.cuh"

// Per-lane, loop-invariant description of what a lane requests from every input row.  A lane owns NW units of
// 16 input bytes (= 8*NW output pixels).  The kernel is only used for w % 16 == 0, so a unit is either fully inside
// the row or starts exactly at w; the reflect-101 halo bytes (p[-1]=p[1], p[-2]=p[2], p[w]=p[w-2], p[w+1]=p[w-3])
// come from one aligned word and a byte permute.
//
// Rows travel global -> shared with cp.async (LDGSTS) into a per-warp ring, PF_Q rows ahead of the row being
// consumed: no registers are tied up by loads in flight, and the halo words of a lane are simply its neighbours'
// words in the ring.  Ring row: [12 pad][4 left halo][32 lanes x 16*NW B][4 right halo][12 pad].
// Every lane executes the same (predicated) requests per row; a size of 0 masks the lane off.
template <int NW>
struct LanePlan {
  int unit_size[NW];         // 16-byte request of unit k is live
  int refl_size, refl_dst;   // the unit that starts exactly at w receives p[w-4..w-1] in its first word
  int edge_off, edge_size, edge_dst;   // 4-byte halo request of lanes 0 / 31
  uint32_t left_sel, right_sel;        // byte_perm selectors of the halo words (identity unless reflecting)
  uint32_t unit_sel[NW];               // selector of the first word of unit k >= 1 (it is unit k-1's right neighbour)
};

template <int NW>
__device__ __forceinline__ LanePlan<NW> make_plan(int ix0, int w, int lane, int xlim) {
  LanePlan<NW> p;
  p.refl_size = 0; p.refl_dst = 0;
#pragma unroll
  for (int k = 0; k < NW; ++k) {
    const int ux = ix0 + 16 * k;
    p.unit_size[k] = (ux + 16 <= w && ux < xlim) ? 16 : 0;   // units past the last stored column's taps are not fetched
    p.unit_sel[k] = ux == w ? 0x4412u : 0x3210u;       // (p[w-2], p[w-3], -, -) from p[w-4..w-1]
    if (ux == w) { p.refl_size = 4; p.refl_dst = 16 + 16 * NW * lane + 16 * k; }
  }
  p.left_sel = ix0 == 0 ? 0x1244u : 0x3210u;           // (-, -, p[2], p[1]) from p[0..3]
  p.right_sel = ix0 + 16 * NW == w ? 0x4412u : 0x3210u;
  p.edge_off = 0; p.edge_size = 0; p.edge_dst = 4;     // bytes 0..11 of a ring row are padding
  if (lane == 0) {
    p.edge_size = 4; p.edge_dst = 12;
    p.edge_off = ix0 >= 4 ? ix0 - 4 : 0;
  } else if (lane == 31 && ix0 + 16 * NW <= w) {
    p.edge_size = 4; p.edge_dst = 16 + 16 * NW * 32;
    p.edge_off = ix0 + 16 * NW + 4 <= w ? ix0 + 16 * NW : w - 4;
  }
  return p;
}

// predicated cp.async: lanes whose request does not apply are masked off (no divergent branch, no smem write)
__device__ __forceinline__ void cp_async16(uint32_t smem, const void* gmem, int size) {
  asm volatile("{ .reg .pred p; setp.ne.s32 p, %2, 0; @p cp.async.cg.shared.global [%0], [%1], 16; }" ::"r"(smem), "l"(gmem), "r"(size));
}
__device__ __forceinline__ void cp_async4(uint32_t smem, const void* gmem, int size) {
  asm volatile("{ .reg .pred p; setp.ne.s32 p, %2, 0; @p cp.async.ca.shared.global [%0], [%1], 4; }" ::"r"(smem), "l"(gmem), "r"(size));
}

// One warp computes output rows [oy0, oy1) x the 8*NW output columns of each lane starting at ox0 (ix0 = 2*ox0 in the
// source, whose width w is a multiple of 16 and whose rows are 16 B aligned); columns >= xo1 (a multiple of 8) are not
// stored.  ring0 = shared-memory address of this warp's ring of (PF_Q + 4) rows of (16 + 16*NW*32 + 16) bytes.
template <int PF_Q, int NW>
__device__ __forceinline__ void agt_pyr_down_strip(const uint8_t* __restrict__ img, int w, int h, int64_t spitch,
                                                   uint8_t* __restrict__ out, int64_t dpitch, int ox0, int xo1, int oy0, int oy1,
                                                   int lane, uint32_t ring0) {
  constexpr int NWORD = 4 * NW;                // own 32-bit words per lane and row
  constexpr int RPITCH = 16 + 16 * NW * 32 + 16;
  constexpr int PF_RING = PF_Q + 4;
  const int ix0 = 2 * ox0;
  const LanePlan<NW> plan = make_plan<NW>(ix0, w, lane, 2 * xo1 + 4);
  const uint32_t ring_end = ring0 + PF_RING * RPITCH;
  const uint32_t lane_main = 16 + 16 * NW * lane;
  const int n_in = 2 * (oy1 - oy0) + 3;            // input rows the strip consumes
  int r_next = 2 * oy0 - 2, issued = 0;            // next input row to request
  uint32_t req_slot = ring0, take_slot = ring0;

  // request one input row (sizes forced to 0 past the end of the strip) and close the group
  auto request = [&]() {
    // BORDER_REFLECT_101 with a single fold: rows overshoot by at most 2 and h >= 4
    int rr = h - 1 - abs(h - 1 - abs(r_next));
    const uint8_t* row = img + (int64_t)rr * spitch;
    const bool live = issued < n_in;
#pragma unroll
    for (int k = 0; k < NW; ++k) cp_async16(req_slot + lane_main + 16 * k, row + ix0 + 16 * k, live ? plan.unit_size[k] : 0);
    cp_async4(req_slot + plan.refl_dst, row + w - 4, live ? plan.refl_size : 0);
    cp_async4(req_slot + plan.edge_dst, row + plan.edge_off, live ? plan.edge_size : 0);
    asm volatile("cp.async.commit_group;");
    ++r_next; ++issued;
    req_slot += RPITCH;
    if (req_slot == ring_end) req_slot = ring0;
  };
  // wait for the oldest outstanding row, read own bytes + the neighbours' halo words, horizontal pass
  auto take = [&](uint32_t hrow[NWORD]) {
    asm volatile("cp.async.wait_group %0;" ::"n"(PF_Q));
    __syncwarp();
    uint32_t wv[NWORD + 2];
    const uint32_t at = take_slot + lane_main;
#pragma unroll
    for (int k = 0; k < NW; ++k)
      asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];"
                   : "=r"(wv[1 + 4 * k]), "=r"(wv[2 + 4 * k]), "=r"(wv[3 + 4 * k]), "=r"(wv[4 + 4 * k]) : "r"(at + 16 * k));
    uint32_t left, right;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(left) : "r"(at - 4));
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(right) : "r"(at + 16 * NW));
    wv[0] = __byte_perm(left, 0u, plan.left_sel);
    wv[NWORD + 1] = __byte_perm(right, 0u, plan.right_sel);
#pragma unroll
    for (int k = 1; k < NW; ++k) wv[1 + 4 * k] = __byte_perm(wv[1 + 4 * k], 0u, plan.unit_sel[k]);
#pragma unroll
    for (int j = 0; j < NWORD; ++j) {
      uint32_t even = __dp4a(wv[j], 0x04010000u, __dp4a(wv[j + 1], 0x00010406u, 0u));
      uint32_t odd = __dp4a(wv[j + 1], 0x04060401u, __dp4a(wv[j + 2], 0x00000001u, 0u));
      hrow[j] = __byte_perm(even, odd, 0x5410);            // even | odd << 16 (both < 65536)
    }
    take_slot += RPITCH;
    if (take_slot == ring_end) take_slot = ring0;
  };
  // vertical [1 4 6 4 1] on packed u16 pairs, +128, >>8, and the four result bytes of two words in one permute
  auto emit = [&](int oy, const uint32_t* a, const uint32_t* b, const uint32_t* c, const uint32_t* d, const uint32_t* e) {
    uint32_t px[NWORD / 2];
#pragma unroll
    for (int j = 0; j < NWORD; j += 2) {
      uint32_t v0 = (a[j] + 4u * (b[j] + d[j])) + (e[j] + 6u * c[j]) + 0x00800080u;
      uint32_t v1 = (a[j + 1] + 4u * (b[j + 1] + d[j + 1])) + (e[j + 1] + 6u * c[j + 1]) + 0x00800080u;
      px[j / 2] = __byte_perm(v0, v1, 0x7531);
    }
    uint8_t* o = out + (int64_t)oy * dpitch + ox0;
    if (NW == 2) {
      if (ox0 + 16 <= xo1) *reinterpret_cast<uint4*>(o) = make_uint4(px[0], px[1], px[2], px[3]);
      else if (ox0 + 8 <= xo1) *reinterpret_cast<uint2*>(o) = make_uint2(px[0], px[1]);
    } else {
      if (ox0 < xo1) *reinterpret_cast<uint2*>(o) = make_uint2(px[0], px[1]);      // xo1 % 8 == 0 on this path
    }
  };

#pragma unroll
  for (int k = 0; k < PF_Q + 1; ++k) request();
  uint32_t h0[NWORD], h1[NWORD], h2[NWORD], h3[NWORD], h4[NWORD], h5[NWORD];
  take(h0); request();
  take(h1); request();
  take(h2); request();
  for (int oy = oy0; oy < oy1; oy += 3) {
    take(h3); request(); take(h4); request();
    emit(oy, h0, h1, h2, h3, h4);
    if (oy + 1 < oy1) {
      take(h5); request(); take(h0); request();
      emit(oy + 1, h2, h3, h4, h5, h0);
    }
    if (oy + 2 < oy1) {
      take(h1); request(); take(h2); request();
      emit(oy + 2, h4, h5, h0, h1, h2);
    }
  }
}
