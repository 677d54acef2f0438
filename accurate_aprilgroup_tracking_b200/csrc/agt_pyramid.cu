// K1: Gaussian pyramid (cv::pyrDown) and Scharr derivatives (cv::Scharr CV_16S),
// integer-exact.  The reference snapshot has no such code; the frozen semantics
// are OpenCV's (SURVEY.md 8a row A5, 9.1): 5x5 [1 4 6 4 1]^2, (sum+128)>>8,
// BORDER_REFLECT_101, output ((w+1)/2, (h+1)/2); Scharr [3 10 3] x [-1 0 1],
// unnormalised int16, BORDER_REFLECT_101.
//
// pyrDown is a pure streaming stencil (HBM-bound): each CTA stages a
// (2*128+32) x (2*16+3) u8 input tile in shared memory with 128-bit coalesced
// loads, runs the horizontal 5-tap pass into a uint16 tile, then the vertical
// pass, and stores 8 output bytes per thread.
#include "agt_common.cuh"
#include "agt_pyr_stream.cuh"

namespace {

constexpr int PD_OW = 128;                 // output tile width
constexpr int PD_OH = 16;                  // output tile height
constexpr int PD_IW = 2 * PD_OW + 32;      // staged input width (16 B aligned start, 16 B slack each side)
constexpr int PD_IH = 2 * PD_OH + 3;
constexpr int PD_THREADS = 256;

__global__ void __launch_bounds__(PD_THREADS)
pyr_down_kernel(const uint8_t* __restrict__ src, int w, int h, int64_t spitch, int64_t sstride,
                uint8_t* __restrict__ dst, int ow, int oh, int64_t dpitch, int64_t dstride, int vec_ok,
                const uint8_t* __restrict__ mask, int mask_stride) {
  if (mask != nullptr) {
    bool any = false;
    for (int k = 0; k < mask_stride; ++k) any = any || mask[(int64_t)blockIdx.z * mask_stride + k] != 0;
    if (!any) return;
  }
  __shared__ __align__(16) uint8_t s_in[PD_IH][PD_IW];
  __shared__ __align__(16) uint16_t s_h[PD_IH][PD_OW];

  const int x0 = blockIdx.x * PD_OW;       // first output column of the tile
  const int y0 = blockIdx.y * PD_OH;
  const uint8_t* img = src + (int64_t)blockIdx.z * sstride;
  uint8_t* out = dst + (int64_t)blockIdx.z * dstride;
  const int gx_base = 2 * x0 - 16;         // global column of s_in[.][0]
  const int gy_base = 2 * y0 - 2;

  // ---- stage the input tile --------------------------------------------------
  constexpr int CHUNKS = PD_IW / 16;
  for (int i = threadIdx.x; i < PD_IH * CHUNKS; i += PD_THREADS) {
    int r = i / CHUNKS, c = i - r * CHUNKS;
    int gy = agt_reflect101(gy_base + r, h);
    int gx = gx_base + 16 * c;
    const uint8_t* row = img + (int64_t)gy * spitch;
    uint4 v;
    if (vec_ok && gx >= 0 && gx + 16 <= w) {
      v = __ldg(reinterpret_cast<const uint4*>(row + gx));
    } else {
      uint32_t word[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        uint32_t acc = 0;
#pragma unroll
        for (int b = 0; b < 4; ++b) {
          int xx = gx + 4 * k + b;
          uint32_t px = row[agt_reflect101(xx, w)];
          acc |= px << (8 * b);
        }
        word[k] = acc;
      }
      v = make_uint4(word[0], word[1], word[2], word[3]);
    }
    *reinterpret_cast<uint4*>(&s_in[r][16 * c]) = v;
  }
  __syncthreads();

  // ---- horizontal pass: 4 outputs per work item ---------------------------------
  // output column x (tile-local, multiple of 4) needs staged bytes 2x+14 .. 2x+24
  constexpr int HGROUPS = PD_OW / 4;
  for (int i = threadIdx.x; i < PD_IH * HGROUPS; i += PD_THREADS) {
    int r = i / HGROUPS, g = i - r * HGROUPS;
    const uint2* p = reinterpret_cast<const uint2*>(&s_in[r][8 * g + 8]);   // bytes 2x+8 .. 2x+31
    uint2 a = p[0], b = p[1], c = p[2];
    // byte k of the 24-byte window = staged byte 2x+8+k ; tap j of output q is byte 6+2q+j
    uint32_t wv[6] = {a.x, a.y, b.x, b.y, c.x, c.y};
    auto byte_at = [&](int k) -> uint32_t { return (wv[k >> 2] >> (8 * (k & 3))) & 0xffu; };
    uint16_t o[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      int k = 6 + 2 * q;
      uint32_t s = byte_at(k) + 4u * byte_at(k + 1) + 6u * byte_at(k + 2) + 4u * byte_at(k + 3) + byte_at(k + 4);
      o[q] = (uint16_t)s;
    }
    uint2 packed = make_uint2((uint32_t)o[0] | ((uint32_t)o[1] << 16), (uint32_t)o[2] | ((uint32_t)o[3] << 16));
    *reinterpret_cast<uint2*>(&s_h[r][4 * g]) = packed;
  }
  __syncthreads();

  // ---- vertical pass: 8 outputs per thread --------------------------------------
  {
    int ty = threadIdx.x / (PD_OW / 8);
    int tx = (threadIdx.x % (PD_OW / 8)) * 8;
    int oy = y0 + ty, ox = x0 + tx;
    if (oy < oh && ox < ow) {
      uint32_t acc[8];
#pragma unroll
      for (int k = 0; k < 8; ++k) acc[k] = 128u;
      const uint32_t wgt[5] = {1u, 4u, 6u, 4u, 1u};
#pragma unroll
      for (int j = 0; j < 5; ++j) {
        uint4 v = *reinterpret_cast<const uint4*>(&s_h[2 * ty + j][tx]);
        uint32_t vv[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          acc[2 * k] += wgt[j] * (vv[k] & 0xffffu);
          acc[2 * k + 1] += wgt[j] * (vv[k] >> 16);
        }
      }
      uint8_t* orow = out + (int64_t)oy * dpitch + ox;
      if (vec_ok && ox + 8 <= ow && ((dpitch & 7) == 0)) {
        uint2 pk;
        pk.x = (acc[0] >> 8) | ((acc[1] >> 8) << 8) | ((acc[2] >> 8) << 16) | ((acc[3] >> 8) << 24);
        pk.y = (acc[4] >> 8) | ((acc[5] >> 8) << 8) | ((acc[6] >> 8) << 16) | ((acc[7] >> 8) << 24);
        *reinterpret_cast<uint2*>(orow) = pk;
      } else {
        for (int k = 0; k < 8 && ox + k < ow; ++k) orow[k] = (uint8_t)(acc[k] >> 8);
      }
    }
  }
}


// ---------------------------------------------------------------------------------------------
// Streaming pyrDown (the hot variant): no shared memory.  A lane owns 8 output columns = 16 input
// bytes per row: one coalesced 128-bit load per input row, the 4-byte halos come from the
// neighbouring lanes by warp shuffle.  The horizontal 5-tap is two dp4a per output, sums are kept
// as packed 2 x u16 (max 16*255 = 4080), the vertical 5-tap runs on the packed words (max
// 16*4080+128 < 65536, so the halves never carry into each other) and each lane stores 8 bytes.
// A warp walks down a strip of PF_STRIP output rows; two new input rows per output row, with the
// next pair of loads issued before the current pair is consumed.
// ---------------------------------------------------------------------------------------------
constexpr int PF_WARPS = 4;

// Streaming pyrDown.  Lane = 8*NW output pixels; horizontal 5-tap = two dp4a per output into packed 2 x u16
// (max 16*255 = 4080); vertical 5-tap on the packed words (max 16*4080+128 < 65536, the halves never carry into each
// other); +128, >>8 and byte packing in one permute per two words; 8*NW-byte stores.  A warp walks down a strip of
// PF_STRIP output rows; six packed row registers rotate with period three output rows, so nothing is ever moved.
template <int PF_Q, int PF_STRIP, int NW, bool kStride>
__global__ void __launch_bounds__(PF_WARPS * 32, NW == 1 ? 6 : 4)
pyr_down_stream_kernel(const uint8_t* __restrict__ src, int w, int h, int64_t spitch, int64_t sstride,
                       uint8_t* __restrict__ dst, int ow, int oh, int64_t dpitch, int64_t dstride,
                       int col_blocks, int strips, int64_t total_warps, const int32_t* __restrict__ rects, int rect_stride,
                       int src_level, const uint8_t* __restrict__ mask, int mask_stride) {
  constexpr int OUTS = 8 * NW;                 // output pixels per lane
  constexpr int RPITCH = 16 + 16 * NW * 32 + 16;
  constexpr int PF_RING = PF_Q + 4;
  const int lane = threadIdx.x & 31;
  __shared__ __align__(16) uint8_t s_ring[PF_WARPS][PF_RING][RPITCH];
  // One work item = one strip of one column block of one frame.  Full-frame and ROI launches have one warp per item;
  // masked launches (few frames flagged, usually none) use a small grid whose warps stride over the items, so that
  // a batch with nothing to redo costs a scan of the mask instead of tens of thousands of empty CTAs.
  if (kStride && mask != nullptr) {
    // nothing flagged in the whole batch (the usual case of the exactness net): leave after one pass over the mask
    const int64_t n_flags = total_warps / ((int64_t)col_blocks * strips) * mask_stride;
    uint32_t acc = 0;
    if ((reinterpret_cast<uintptr_t>(mask) & 15) == 0) {
      const uint4* m4 = reinterpret_cast<const uint4*>(mask);
#pragma unroll 4
      for (int64_t i = threadIdx.x; i < n_flags / 16; i += blockDim.x) { const uint4 v = __ldg(m4 + i); acc |= v.x | v.y | v.z | v.w; }
      for (int64_t i = (n_flags & ~15LL) + threadIdx.x; i < n_flags; i += blockDim.x) acc |= mask[i];
    } else {
      for (int64_t i = threadIdx.x; i < n_flags; i += blockDim.x) acc |= mask[i];
    }
    if (!__syncthreads_or(acc != 0)) return;
  }
#define AGT_ITEM_DONE { if (kStride) { wi += (int64_t)gridDim.x * PF_WARPS; __syncwarp(); continue; } else return; }
  for (int64_t wi = (int64_t)blockIdx.x * PF_WARPS + (threadIdx.x >> 5);;) {
  if (wi >= total_warps) return;
  int64_t wg = wi;
  const int cb = (int)(wg % col_blocks);
  wg /= col_blocks;
  const int strip = (int)(wg % strips);
  const int64_t frame = wg / strips;
  if (mask != nullptr) {                      // only frames with a set flag (any of mask_stride entries)
    bool any = false;
    for (int k = 0; k < mask_stride; ++k) any = any || mask[frame * mask_stride + k] != 0;
    if (!any) AGT_ITEM_DONE;
  }
  // output window of this frame: the whole level, or the part of it below the frame's level-0 rectangle
  int xo0 = 0, yo0 = 0, xo1 = ow, yo1 = oh;
  if (rects != nullptr) {
    const int32_t* r = rects + frame * rect_stride;
    const int sh = src_level + 1, rnd = (1 << sh) - 1;
    xo0 = max(0, (r[0] >> sh) - 2) & ~(OUTS - 1);
    yo0 = max(0, (r[1] >> sh) - 2);
    xo1 = min(ow, (((r[2] + rnd) >> sh) + 2 + 7) & ~7);
    yo1 = min(oh, ((r[3] + rnd) >> sh) + 2);
    if (r[2] <= r[0] || r[3] <= r[1]) AGT_ITEM_DONE;
  }
  const uint8_t* img = src + frame * sstride;
  uint8_t* out = dst + frame * dstride;
  const int ox0 = xo0 + cb * (32 * OUTS) + lane * OUTS;
  const int oy0 = yo0 + strip * PF_STRIP;
  const int oy1 = min(oy0 + PF_STRIP, yo1);
  if (oy0 >= yo1 || xo0 + cb * (32 * OUTS) >= xo1) AGT_ITEM_DONE;      // warp-uniform

  agt_pyr_down_strip<PF_Q, NW>(img, w, h, spitch, out, dpitch, ox0, xo1, oy0, oy1, lane,
                               (uint32_t)__cvta_generic_to_shared(&s_ring[threadIdx.x >> 5][0][0]));
  AGT_ITEM_DONE;
  }
#undef AGT_ITEM_DONE
}

// Region-of-interest pyramid of a batch in ONE launch: a CTA per frame walks down the levels, its four warps share the rows
// of the frame's window at each level (one strip per warp, so the warps finish together) and meet at a barrier before the
// next level reads what they wrote (from L2).  Per-level launches leave most of the machine idle on these small windows:
// a 600 x 580 rectangle is 10 + 5 + 3 strips per frame, three short launches with their tails, each warp striding over a
// handful of live items (profiles/r01_ncu_pyr_roi.txt).  Same streaming warp routine, same bits.
// (Whole frames through this scheme run as fast as the per-level launches, 1.29 against 1.28 ms per 2048 frames, and a
// 16-warp CTA per SM - fewer frames in flight, so that a level might still be in L2 when the next one reads it - is
// slower, 1.34 ms: whole-frame builds keep the per-level launches.)
template <int Q2, int Q1>
__global__ void __launch_bounds__(PF_WARPS * 32, 4)
pyr_roi_chain_kernel(agt_pyramid pyr, const int32_t* __restrict__ rects, int rect_stride, int batch, uint32_t wide_mask) {
  constexpr int RPITCH2 = 16 + 16 * 2 * 32 + 16, RING2 = Q2 + 4, RPITCH1 = 16 + 16 * 32 + 16, RING1 = Q1 + 4;
  constexpr int RING_BYTES = RPITCH2 * RING2 > RPITCH1 * RING1 ? RPITCH2 * RING2 : RPITCH1 * RING1;
  __shared__ __align__(16) uint8_t s_ring[PF_WARPS][RING_BYTES];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const uint32_t ring0 = (uint32_t)__cvta_generic_to_shared(&s_ring[wid][0]);
  for (int frame = blockIdx.x; frame < batch; frame += gridDim.x) {
    const int32_t* r = rects + (int64_t)frame * rect_stride;
    const int r0 = r[0], r1 = r[1], r2 = r[2], r3 = r[3];
    if (r2 <= r0 || r3 <= r1) continue;                    // (the whole CTA)
    for (int l = 1; l < pyr.levels; ++l) {
      const int w = pyr.width[l - 1], h = pyr.height[l - 1], ow = pyr.width[l], oh = pyr.height[l];
      const int rnd = (1 << l) - 1;
      // the window of pyr_down_stream_kernel for src_level = l - 1; windows of up to 256 pixels fit the 32 lanes at 8 pixels
      // per lane, which costs half the instructions per row of the 16-pixel variant
      const int xo1 = min(ow, (((r2 + rnd) >> l) + 2 + 7) & ~7), yo1 = min(oh, ((r3 + rnd) >> l) + 2);
      const int xlo = max(0, (r0 >> l) - 2), yo0 = max(0, (r1 >> l) - 2);
      const bool wide = ((wide_mask >> l) & 1u) && xo1 - (xlo & ~7) > 256;
      const int outs = wide ? 16 : 8;
      const int xo0 = xlo & ~(outs - 1);
      const uint8_t* img = pyr.data[l - 1] + (int64_t)frame * pyr.frame_stride[l - 1];
      uint8_t* out = pyr.data[l] + (int64_t)frame * pyr.frame_stride[l];
      const int per = (yo1 - yo0 + PF_WARPS - 1) / PF_WARPS;
      const int oy0 = yo0 + wid * per, oy1 = min(oy0 + per, yo1);
      if (oy0 < oy1) {
        for (int bx = xo0; bx < xo1; bx += 32 * outs) {
          if (wide) agt_pyr_down_strip<Q2, 2>(img, w, h, pyr.pitch[l - 1], out, pyr.pitch[l], bx + lane * 16, xo1, oy0, oy1, lane, ring0);
          else      agt_pyr_down_strip<Q1, 1>(img, w, h, pyr.pitch[l - 1], out, pyr.pitch[l], bx + lane * 8, xo1, oy0, oy1, lane, ring0);
          __syncwarp();
        }
      }
      __syncthreads();                                     // level l of this frame is complete (and visible) before level l + 1 reads it
    }
  }
}

// Scharr: one thread per pixel pair; loads go through L1.  Not on the hot path
// (the LK and refinement kernels derive gradients on the fly from the u8 levels);
// exported so the derivative planes themselves can be checked bit-exactly.
__global__ void scharr_kernel(const uint8_t* __restrict__ src, int w, int h, int64_t spitch, int64_t sstride,
                              int16_t* __restrict__ dst) {
  int x = blockIdx.x * blockDim.x + threadIdx.x;
  int y = blockIdx.y * blockDim.y + threadIdx.y;
  if (x >= w || y >= h) return;
  const uint8_t* img = src + (int64_t)blockIdx.z * sstride;
  int xm = agt_reflect101(x - 1, w), xp = agt_reflect101(x + 1, w);
  int ym = agt_reflect101(y - 1, h), yp = agt_reflect101(y + 1, h);
  const uint8_t* r0 = img + (int64_t)ym * spitch;
  const uint8_t* r1 = img + (int64_t)y * spitch;
  const uint8_t* r2 = img + (int64_t)yp * spitch;
  int a00 = r0[xm], a01 = r0[x], a02 = r0[xp];
  int a10 = r1[xm], a12 = r1[xp];
  int a20 = r2[xm], a21 = r2[x], a22 = r2[xp];
  int dx = 3 * (a02 - a00) + 10 * (a12 - a10) + 3 * (a22 - a20);
  int dy = 3 * (a20 - a00) + 10 * (a21 - a01) + 3 * (a22 - a02);
  int16_t* o = dst + ((int64_t)blockIdx.z * h * w + (int64_t)y * w + x) * 2;
  *reinterpret_cast<short2*>(o) = make_short2((short)dx, (short)dy);
}

// Frame ingest (SURVEY.md 8f row N2): cv::cvtColor(BGR2GRAY) for 8-bit images in OpenCV's fixed-point form,
// gray = (B*3735 + G*19235 + R*9798 + 16384) >> 15, written straight into level 0 of a pyramid.
// 16 pixels per thread: three 128-bit loads of interleaved BGR, one 128-bit store.
__global__ void bgr_to_gray_kernel(const uint8_t* __restrict__ bgr, int w, int h, int64_t spitch, int64_t sstride,
                                   uint8_t* __restrict__ gray, int64_t dpitch, int64_t dstride, int vec_ok) {
  const int x0 = (blockIdx.x * blockDim.x + threadIdx.x) * 16;
  const int y = blockIdx.y;
  if (x0 >= w) return;
  const uint8_t* src = bgr + (int64_t)blockIdx.z * sstride + (int64_t)y * spitch + 3 * x0;
  uint8_t* dst = gray + (int64_t)blockIdx.z * dstride + (int64_t)y * dpitch + x0;
  if (vec_ok && x0 + 16 <= w) {
    const uint4* p = reinterpret_cast<const uint4*>(src);
    uint4 q[3] = {__ldg(p), __ldg(p + 1), __ldg(p + 2)};
    const uint32_t* wds = reinterpret_cast<const uint32_t*>(q);
    uint32_t o[4];
#pragma unroll
    for (int g = 0; g < 4; ++g) {            // 4 pixels = 12 bytes = words 3g .. 3g+2
      const uint32_t a = wds[3 * g], b = wds[3 * g + 1], c = wds[3 * g + 2];
      // pixel 0: a.b0 a.b1 a.b2 | pixel 1: a.b3 b.b0 b.b1 | pixel 2: b.b2 b.b3 c.b0 | pixel 3: c.b1 c.b2 c.b3
      const uint32_t px[4] = {a & 0xffffffu, (a >> 24) | ((b & 0xffffu) << 8), (b >> 16) | ((c & 0xffu) << 16), c >> 8};
      uint32_t out = 0;
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const uint32_t B = px[k] & 0xffu, G = (px[k] >> 8) & 0xffu, R = (px[k] >> 16) & 0xffu;
        out |= ((B * 3735u + G * 19235u + R * 9798u + 16384u) >> 15) << (8 * k);
      }
      o[g] = out;
    }
    *reinterpret_cast<uint4*>(dst) = make_uint4(o[0], o[1], o[2], o[3]);
  } else {
    for (int k = 0; k < 16 && x0 + k < w; ++k) {
      const uint32_t B = src[3 * k], G = src[3 * k + 1], R = src[3 * k + 2];
      dst[k] = (uint8_t)((B * 3735u + G * 19235u + R * 9798u + 16384u) >> 15);
    }
  }
}

}  // namespace

extern "C" int agt_bgr_to_gray(agt_ctx* ctx, const uint8_t* d_bgr, int w, int h, int64_t src_pitch, int64_t src_stride,
                               uint8_t* d_gray, int64_t dst_pitch, int64_t dst_stride, int batch) {
  if (!ctx) return AGT_ERR_INVALID;
  if (batch == 0) return AGT_OK;          // nothing to do (empty tensors may carry null pointers)
  if (!d_bgr || !d_gray || w < 1 || h < 1 || batch < 0 || src_pitch < 3 * (int64_t)w || dst_pitch < w)
    AGT_FAIL(ctx, AGT_ERR_INVALID, "agt_bgr_to_gray: bad arguments");
  if (batch == 0) return AGT_OK;
  int vec_ok = ((reinterpret_cast<uintptr_t>(d_bgr) & 15) == 0) && ((src_pitch & 15) == 0) && ((src_stride & 15) == 0) &&
               ((reinterpret_cast<uintptr_t>(d_gray) & 15) == 0) && ((dst_pitch & 15) == 0) && ((dst_stride & 15) == 0);
  for (int b0 = 0; b0 < batch; b0 += 65535) {
    int nb = batch - b0 < 65535 ? batch - b0 : 65535;
    dim3 grid(((w + 15) / 16 + 127) / 128, h, nb);
    bgr_to_gray_kernel<<<grid, 128, 0, ctx->stream>>>(d_bgr + (int64_t)b0 * src_stride, w, h, src_pitch, src_stride,
                                                      d_gray + (int64_t)b0 * dst_stride, dst_pitch, dst_stride, vec_ok);
    AGT_LAUNCH_CHECK(ctx);
  }
  return AGT_OK;
}

static int pyr_down_impl(agt_ctx* ctx, const uint8_t* d_src, int w, int h, int64_t src_pitch, int64_t src_stride,
                         uint8_t* d_dst, int64_t dst_pitch, int64_t dst_stride, int batch, const int32_t* d_rects,
                         int rect_stride, int src_level, const uint8_t* d_mask, int mask_stride) {
  if (batch == 0) return AGT_OK;
  if (!d_src || !d_dst || w < 1 || h < 1 || batch < 0 || src_pitch < w || dst_pitch < (w + 1) / 2)
    AGT_FAIL(ctx, AGT_ERR_INVALID, "agt_pyr_down: bad arguments (w=%d h=%d batch=%d)", w, h, batch);
  if (batch == 0) return AGT_OK;
  int ow = (w + 1) / 2, oh = (h + 1) / 2;
  int vec_ok = ((reinterpret_cast<uintptr_t>(d_src) & 15) == 0) && ((src_pitch & 15) == 0) && ((src_stride & 15) == 0) &&
               ((reinterpret_cast<uintptr_t>(d_dst) & 7) == 0) && ((dst_stride & 7) == 0);
  // streaming kernel: 16 B aligned rows and w % 16 == 0 (every pyramid level of 1080p / VGA); else the tiled kernel
  const bool stream_ok = vec_ok && ((dst_pitch & 7) == 0) && (w & 15) == 0 && w >= 16 && h >= 4;
  if (stream_ok) {
    // wide levels use 16 output pixels per lane (half the per-byte instruction overhead), narrow ones 8
    const bool wide = ow >= 320 && ((dst_pitch & 15) == 0) && ((reinterpret_cast<uintptr_t>(d_dst) & 15) == 0) && ((dst_stride & 15) == 0);
    constexpr int kStrip = 32;
    const int lane_outs = wide ? 16 : 8;
    int col_blocks = (ow + 32 * lane_outs - 1) / (32 * lane_outs), strips = (oh + kStrip - 1) / kStrip;
    int64_t total_warps = (int64_t)batch * strips * col_blocks;
    int64_t blocks = (total_warps + PF_WARPS - 1) / PF_WARPS;
    // Masked launches (few frames flagged) and region-of-interest launches (most items of a level lie outside the frame's
    // rectangle) use a grid that just fills the machine; its warps stride over the items, so every resident warp keeps
    // finding real strips instead of whole CTAs holding their slots for one live warp.
    const int64_t fill = (int64_t)(d_mask != nullptr ? 8 : (wide ? 4 : 6)) * ctx->sm_count;
    const bool stride_items = (d_mask != nullptr || d_rects != nullptr) && blocks > fill;
    if (stride_items) blocks = fill;
    if (blocks <= 0x7fffffffLL) {
#define AGT_PYR_LAUNCH(Q, NWv, ST)                                                                                        \
  pyr_down_stream_kernel<Q, kStrip, NWv, ST><<<(unsigned)blocks, PF_WARPS * 32, 0, ctx->stream>>>(                          \
      d_src, w, h, src_pitch, src_stride, d_dst, ow, oh, dst_pitch, dst_stride, col_blocks, strips, total_warps, d_rects, \
      rect_stride, src_level, d_mask, mask_stride)
      if (wide) { if (stride_items) AGT_PYR_LAUNCH(6, 2, true); else AGT_PYR_LAUNCH(6, 2, false); }
      else      { if (stride_items) AGT_PYR_LAUNCH(8, 1, true); else AGT_PYR_LAUNCH(8, 1, false); }
#undef AGT_PYR_LAUNCH
      AGT_LAUNCH_CHECK(ctx);
      return AGT_OK;
    }
  }
  // tiled kernel (any size / alignment): computes whole frames, which is a superset of any ROI
  for (int b0 = 0; b0 < batch; b0 += 65535) {
    int nb = batch - b0 < 65535 ? batch - b0 : 65535;
    dim3 grid((ow + PD_OW - 1) / PD_OW, (oh + PD_OH - 1) / PD_OH, nb);
    pyr_down_kernel<<<grid, PD_THREADS, 0, ctx->stream>>>(d_src + (int64_t)b0 * src_stride, w, h, src_pitch, src_stride,
                                                          d_dst + (int64_t)b0 * dst_stride, ow, oh, dst_pitch,
                                                          dst_stride, vec_ok, d_mask ? d_mask + (int64_t)b0 * mask_stride : nullptr,
                                                          mask_stride);
    AGT_LAUNCH_CHECK(ctx);
  }
  return AGT_OK;
}

extern "C" int agt_pyr_down(agt_ctx* ctx, const uint8_t* d_src, int w, int h, int64_t src_pitch, int64_t src_stride,
                            uint8_t* d_dst, int64_t dst_pitch, int64_t dst_stride, int batch) {
  if (!ctx) return AGT_ERR_INVALID;
  return pyr_down_impl(ctx, d_src, w, h, src_pitch, src_stride, d_dst, dst_pitch, dst_stride, batch, nullptr, 0, 0, nullptr, 0);
}

static int build_pyramid_impl(agt_ctx* ctx, const agt_pyramid* pyr, int batch, const int32_t* d_rects, int rect_stride,
                              const uint8_t* d_mask, int mask_stride) {
  if (!pyr || pyr->levels < 1 || pyr->levels > AGT_MAX_LEVELS)
    AGT_FAIL(ctx, AGT_ERR_INVALID, "agt_build_pyramid: bad pyramid descriptor");
  // region-of-interest builds of batches that fill the machine: all levels in one launch, a CTA per frame
  if (d_rects != nullptr && d_mask == nullptr && batch >= 2 * ctx->sm_count && pyr->levels > 1) {
    bool ok = true;
    uint32_t wide_mask = 0;
    for (int l = 1; l < pyr->levels && ok; ++l) {
      const int w = pyr->width[l - 1], h = pyr->height[l - 1], ow = pyr->width[l];
      ok = pyr->data[l - 1] && pyr->data[l] && ow == (w + 1) / 2 && pyr->height[l] == (h + 1) / 2 && (w & 15) == 0 && w >= 16 && h >= 4 &&
           ((reinterpret_cast<uintptr_t>(pyr->data[l - 1]) | (uintptr_t)pyr->pitch[l - 1] | (uintptr_t)pyr->frame_stride[l - 1]) & 15) == 0 &&
           ((reinterpret_cast<uintptr_t>(pyr->data[l]) | (uintptr_t)pyr->pitch[l] | (uintptr_t)pyr->frame_stride[l]) & 7) == 0 &&
           pyr->pitch[l - 1] >= w && pyr->pitch[l] >= ow;
      const bool wide = ow >= 320 && ((reinterpret_cast<uintptr_t>(pyr->data[l]) | (uintptr_t)pyr->pitch[l] | (uintptr_t)pyr->frame_stride[l]) & 15) == 0;
      if (wide) wide_mask |= 1u << l;
    }
    if (ok) {
      if (batch == 0) return AGT_OK;
      const int blocks = batch < 4 * ctx->sm_count ? batch : 4 * ctx->sm_count;
      pyr_roi_chain_kernel<6, 8><<<blocks, PF_WARPS * 32, 0, ctx->stream>>>(*pyr, d_rects, rect_stride, batch, wide_mask);
      AGT_LAUNCH_CHECK(ctx);
      return AGT_OK;
    }
  }
  for (int l = 1; l < pyr->levels; ++l) {
    if (pyr->width[l] != (pyr->width[l - 1] + 1) / 2 || pyr->height[l] != (pyr->height[l - 1] + 1) / 2)
      AGT_FAIL(ctx, AGT_ERR_INVALID, "agt_build_pyramid: level %d is not ((w+1)/2,(h+1)/2) of level %d", l, l - 1);
    int rc = pyr_down_impl(ctx, pyr->data[l - 1], pyr->width[l - 1], pyr->height[l - 1], pyr->pitch[l - 1],
                           pyr->frame_stride[l - 1], pyr->data[l], pyr->pitch[l], pyr->frame_stride[l], batch, d_rects,
                           rect_stride, l - 1, d_mask, mask_stride);
    if (rc != AGT_OK) return rc;
  }
  return AGT_OK;
}

extern "C" int agt_build_pyramid(agt_ctx* ctx, const agt_pyramid* pyr, int batch) {
  if (!ctx) return AGT_ERR_INVALID;
  return build_pyramid_impl(ctx, pyr, batch, nullptr, 0, nullptr, 0);
}

extern "C" int agt_build_pyramid_roi(agt_ctx* ctx, const agt_pyramid* pyr, const int32_t* d_rects, int rect_stride, int batch) {
  if (!ctx) return AGT_ERR_INVALID;
  if (!d_rects || rect_stride < 4) AGT_FAIL(ctx, AGT_ERR_INVALID, "agt_build_pyramid_roi: rects missing or rect_stride < 4");
  return build_pyramid_impl(ctx, pyr, batch, d_rects, rect_stride, nullptr, 0);
}

extern "C" int agt_build_pyramid_masked(agt_ctx* ctx, const agt_pyramid* pyr, const uint8_t* d_mask, int mask_stride, int batch) {
  if (!ctx) return AGT_ERR_INVALID;
  if (!d_mask || mask_stride < 1) AGT_FAIL(ctx, AGT_ERR_INVALID, "agt_build_pyramid_masked: mask missing");
  return build_pyramid_impl(ctx, pyr, batch, nullptr, 0, d_mask, mask_stride);
}

extern "C" int agt_scharr(agt_ctx* ctx, const uint8_t* d_src, int w, int h, int64_t src_pitch, int64_t src_stride,
                          int16_t* d_dst, int batch) {
  if (!ctx) return AGT_ERR_INVALID;
  if (batch == 0) return AGT_OK;          // nothing to do (empty tensors may carry null pointers)
  if (!d_src || !d_dst || w < 1 || h < 1 || batch < 0 || src_pitch < w)
    AGT_FAIL(ctx, AGT_ERR_INVALID, "agt_scharr: bad arguments");
  if (batch == 0) return AGT_OK;
  dim3 block(32, 8);
  for (int b0 = 0; b0 < batch; b0 += 65535) {
    int nb = batch - b0 < 65535 ? batch - b0 : 65535;
    dim3 grid((w + 31) / 32, (h + 7) / 8, nb);
    scharr_kernel<<<grid, block, 0, ctx->stream>>>(d_src + (int64_t)b0 * src_stride, w, h, src_pitch, src_stride,
                                                   d_dst + (int64_t)b0 * h * w * 2);
    AGT_LAUNCH_CHECK(ctx);
  }
  return AGT_OK;
}
