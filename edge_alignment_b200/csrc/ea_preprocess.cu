// Frame preprocessing kernels (sm_100a), batched over n frames.
//
// Replaces the OpenCV call sequences of
//   get_aX                  standalone/utils.cpp:201-281  (GaussianBlur, cvtColor, Laplacian, convertScaleAbs,
//                                                          threshold, Z>0 test, row-major ordered compaction)
//   get_distance_transform  standalone/utils.cpp:38-83    (same gradient, medianBlur 3, distanceTransform(L2,3),
//                                                          normalize MINMAX)
// Integer stages are bit-exact restatements of OpenCV's portable code paths (pinned in tests/golden).
// HBM-bound byte/integer work: coalesced loads, shared-memory staging, no tensor cores.
#include <cstdlib>
#include <cstring>

#include "ea_internal.h"

namespace {

__device__ __forceinline__ int reflect101(int i, int n) {
  if (n == 1) return 0;
  while (i < 0 || i >= n) i = (i < 0) ? -i : 2 * n - 2 - i;
  return i;
}

// ---- pyramid: cv::resize(0.5) INTER_LINEAR on BGR or gray (== 2x2 mean, +2 >> 2, per channel), INTER_NEAREST on depth
// CN: channels of the image (3: BGR, 1: gray).  A one-channel source is read where it lies (EaImage: the caller's luma at level
// 0); the depth source is dense, src_frame_stride_px pixels per frame.
template <typename D, int CN>
__global__ void __launch_bounds__(256) k_pyr_down(const EaImage src, const D* __restrict__ src_depth,
                                                  size_t src_frame_stride_px, const int32_t* __restrict__ src_slots,
                                                  uint8_t* __restrict__ dst_bgr, D* __restrict__ dst_depth,
                                                  const int32_t* __restrict__ dst_slots, int sw, int sh) {
  const int dw = sw >> 1, dh = sh >> 1;
  const int f = blockIdx.y;
  const size_t sf = src_slots ? size_t(src_slots[f]) : size_t(f);
  const size_t sbase = sf * src_frame_stride_px;
  const size_t dbase = size_t(dst_slots[f]) * size_t(dw) * dh;
  const uint8_t* src_bgr = src.base;
  const uint8_t* fr = src.base + sf * src.stride + src.offset;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < dw * dh; i += gridDim.x * blockDim.x) {
    const int x = i % dw, y = i / dw;
    uint8_t* d = dst_bgr + (dbase + i) * CN;
    if constexpr (CN == 3) {
      const uint8_t* p = src_bgr + (sbase + size_t(2 * y) * sw + 2 * x) * CN;
      const uint8_t* q = p + size_t(sw) * CN;
#pragma unroll
      for (int c = 0; c < CN; ++c) d[c] = uint8_t((p[c] + p[CN + c] + q[c] + q[CN + c] + 2) >> 2);
    } else {
      const uint8_t* p = fr + size_t(2 * y) * src.pitch + size_t(2 * x) * src.step;
      const uint8_t* q = p + src.pitch;
      d[0] = uint8_t((p[0] + p[src.step] + q[0] + q[src.step] + 2) >> 2);
    }
    if (src_depth) dst_depth[dbase + i] = src_depth[sbase + size_t(2 * y) * sw + 2 * x];
  }
}

// Same arithmetic, four output pixels per thread: 2 x 8 CN source bytes as 8-byte loads, 4 CN result bytes as 4-byte stores
// (the byte-per-load version above moves 3.3 TB/s on BGR; frames whose rows allow it take this one).  Needs dw % 4 == 0 and
// 8-byte aligned frame bases; one-channel input: planar, with 8-byte aligned rows.
template <typename D, int CN>
__global__ void __launch_bounds__(256) k_pyr_down4(const EaImage src, const D* __restrict__ src_depth,
                                                   size_t src_frame_stride_px, const int32_t* __restrict__ src_slots,
                                                   uint8_t* __restrict__ dst_bgr, D* __restrict__ dst_depth,
                                                   const int32_t* __restrict__ dst_slots, int sw, int sh) {
  const int dw = sw >> 1, dh = sh >> 1, qw = dw >> 2;
  const int f = blockIdx.y;
  const size_t sf = src_slots ? size_t(src_slots[f]) : size_t(f);
  const size_t sbase = sf * src_frame_stride_px;
  const size_t dbase = size_t(dst_slots[f]) * size_t(dw) * dh;
  const uint8_t* src_bgr = src.base;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < qw * dh; i += gridDim.x * blockDim.x) {
    const int xq = i % qw, y = i / qw;
    const uint2 *p, *q;
    if constexpr (CN == 3) {
      p = reinterpret_cast<const uint2*>(src_bgr + (sbase + size_t(2 * y) * sw + size_t(8 * xq)) * CN);
      q = reinterpret_cast<const uint2*>(src_bgr + (sbase + size_t(2 * y + 1) * sw + size_t(8 * xq)) * CN);
    } else {
      p = reinterpret_cast<const uint2*>(src.base + sf * src.stride + size_t(2 * y) * src.pitch + size_t(8 * xq));
      q = reinterpret_cast<const uint2*>(reinterpret_cast<const uint8_t*>(p) + src.pitch);
    }
    union { uint2 v[CN]; unsigned char b[8 * CN]; } a, c;
#pragma unroll
    for (int k = 0; k < CN; ++k) { a.v[k] = __ldg(p + k); c.v[k] = __ldg(q + k); }
    union { unsigned w[CN]; unsigned char b[4 * CN]; } o;
#pragma unroll
    for (int px = 0; px < 4; ++px)
#pragma unroll
      for (int ch = 0; ch < CN; ++ch)
        o.b[CN * px + ch] = (unsigned char)((a.b[2 * CN * px + ch] + a.b[2 * CN * px + CN + ch] + c.b[2 * CN * px + ch] + c.b[2 * CN * px + CN + ch] + 2) >> 2);
    unsigned* d = reinterpret_cast<unsigned*>(dst_bgr + (dbase + size_t(y) * dw + size_t(4 * xq)) * CN);
#pragma unroll
    for (int k = 0; k < CN; ++k) d[k] = o.w[k];
    if (src_depth) {
#pragma unroll
      for (int px = 0; px < 4; ++px) dst_depth[dbase + size_t(y) * dw + 4 * xq + px] = src_depth[sbase + size_t(2 * y) * sw + 2 * (4 * xq + px)];
    }
  }
}

// ---- fused GaussianBlur3 -> RGB2GRAY -> Laplacian3 -> |.| saturate -> threshold -> bit mask ----------------
// Block = 32x8 pixels; one ballot word per warp row.  CN = 1: gray input, blurred straight into the gray tile (RGB2GRAY of
// three equal channels is the identity: 9798 + 19235 + 3735 == 1 << 15).
#define ET_W 32
#define ET_H 8
// CN = 1: the image is read where it lies (EaImage); depth is dense, frame_stride_px pixels per frame.
template <typename D, int CN>
__global__ void __launch_bounds__(256) k_edge_mask(const EaImage img, const D* __restrict__ depth,
                                                   size_t frame_stride_px, const int32_t* __restrict__ src_slots,
                                                   const int32_t* __restrict__ dst_slots, uint32_t* __restrict__ edge_bits,
                                                   uint32_t* __restrict__ ref_bits, int w, int h, int words, int thresh, int zero_to_one) {
  __shared__ uint8_t tile[ET_H + 4][(ET_W + 4) * CN + 4];
  __shared__ uint8_t gray[ET_H + 2][ET_W + 2 + 2];
  const int f = blockIdx.z;
  const size_t sf = src_slots ? size_t(src_slots[f]) : size_t(f);
  const size_t sbase = sf * frame_stride_px;
  const uint8_t* bgr = img.base;
  const uint8_t* fr = img.base + sf * img.stride + img.offset;
  const int x0 = blockIdx.x * ET_W, y0 = blockIdx.y * ET_H;
  const int tid = threadIdx.y * ET_W + threadIdx.x;
  // stage the tile with a 2-pixel halo; outside the image map through REFLECT_101 (the composition of the
  // blur's and the Laplacian's border handling reduces to this because both kernels are symmetric)
  for (int i = tid; i < (ET_H + 4) * (ET_W + 4) * CN; i += 256) {
    const int row = i / ((ET_W + 4) * CN), b = i % ((ET_W + 4) * CN);
    const int px = b / CN, c = b % CN;
    const int gx = reflect101(x0 - 2 + px, w), gy = reflect101(y0 - 2 + row, h);
    if constexpr (CN == 3) tile[row][b] = bgr[(sbase + size_t(gy) * w + gx) * CN + c];
    else tile[row][b] = fr[size_t(gy) * img.pitch + size_t(gx) * img.step];
  }
  __syncthreads();
  for (int i = tid; i < (ET_H + 2) * (ET_W + 2); i += 256) {
    const int gyr = i / (ET_W + 2), gxr = i % (ET_W + 2);  // gray position == tile position (gxr+1, gyr+1)
    int ch[CN];
#pragma unroll
    for (int c = 0; c < CN; ++c) {
      const uint8_t* r0 = &tile[gyr][gxr * CN + c];
      const uint8_t* r1 = &tile[gyr + 1][gxr * CN + c];
      const uint8_t* r2 = &tile[gyr + 2][gxr * CN + c];
      const int s = (r0[0] + 2 * r0[CN] + r0[2 * CN]) + 2 * (r1[0] + 2 * r1[CN] + r1[2 * CN]) + (r2[0] + 2 * r2[CN] + r2[2 * CN]);
      ch[c] = (s + 8) >> 4;                       // GaussianBlur 3x3 sigma 0: [1 2 1]/4 separable, one rounding
    }
    if constexpr (CN == 3) gray[gyr][gxr] = uint8_t((ch[0] * 9798 + ch[1] * 19235 + ch[2] * 3735 + 16384) >> 15);  // RGB2GRAY on BGR data
    else gray[gyr][gxr] = uint8_t(ch[0]);
  }
  __syncthreads();
  const int lx = threadIdx.x, ly = threadIdx.y, x = x0 + lx, y = y0 + ly;
  bool edge = false, valid = false;
  if (x < w && y < h) {
    const int gx = lx + 1, gy = ly + 1;
    int v = 2 * (gray[gy - 1][gx - 1] + gray[gy - 1][gx + 1] + gray[gy + 1][gx - 1] + gray[gy + 1][gx + 1]) - 8 * gray[gy][gx];
    v = v < 0 ? -v : v;                             // Laplacian ksize 3 + convertScaleAbs
    edge = min(v, 255) > thresh;
    if (depth) valid = zero_to_one || depth[sbase + size_t(y) * w + x] > D(0);
  }
  const unsigned eb = __ballot_sync(0xffffffffu, edge);
  const unsigned rb = __ballot_sync(0xffffffffu, edge && valid);
  if (lx == 0 && y < h) {
    const size_t o = (size_t(dst_slots[f]) * h + y) * words + blockIdx.x;
    edge_bits[o] = eb;
    if (ref_bits) ref_bits[o] = rb;
  }
}

// ---- v2 of the fused edge kernel: 128x32 output tile per CTA, packed pixels, separable rolling windows --------
// Same arithmetic as k_edge_mask (bit exact); ~3x fewer instructions per pixel.  Needs w % 4 == 0 (32-bit row loads).
#define E2_TW 128
#define E2_TH 32
#define E2_PH (E2_TH + 4)   // image rows y0-2 .. y0+33 (through REFLECT_101)

// packed pixel p = B | G<<8 | R<<16  ->  16-bit lanes {B, G} and {R}
__device__ __forceinline__ void e2_expand(unsigned p, unsigned& bg, unsigned& r) {
  bg = __byte_perm(p, 0, 0x4140);
  r = __byte_perm(p, 0, 0x4442);
}
// 3x3 Gaussian rounding + RGB2GRAY (on BGR data) from vertical sums held in 16-bit lanes
__device__ __forceinline__ unsigned e2_gray(unsigned v_bg, unsigned v_r) {
  const unsigned b_bg = ((v_bg + 0x00080008u) >> 4) & 0x00FF00FFu;
  const unsigned b_r = (v_r + 8u) >> 4;
  const unsigned B = b_bg & 0xFFFFu, G = b_bg >> 16;
  return (B * 9798u + G * 19235u + b_r * 3735u + 16384u) >> 15;
}

// Phase 3 of the fused edge kernels: Laplacian (ksize 3) + convertScaleAbs + threshold over the gray tile (column g <-> image
// column x0 - 1 + g, row r <-> image row y0 - 1 + r), one ballot word per warp row; REF: also the reference-point plane.
// min(|v|, 255) > thresh  <=>  |v| > thresh for thresh < 255 (never true above); columns beyond the image read gray
// column 0 (harmless) and vote "no edge"; the row loop stops at the image's last row.
template <typename D, int TW, bool REF>
__device__ __forceinline__ void e2_laplacian_bits(const uint8_t (*gray)[TW + 4], const D* __restrict__ depth, size_t sbase, int dst_slot,
                                                  uint32_t* __restrict__ edge_bits, uint32_t* __restrict__ ref_bits, int x0, int y0,
                                                  int w, int h, int words, int thresh, int zero_to_one) {
  const int t = threadIdx.x;
  const int x = x0 + t, lane = t & 31, wq = t >> 5;
  const bool col_ok = x < w;
  const int gl = col_ok ? reflect101(x - 1, w) - x0 + 1 : 0, gc = col_ok ? t + 1 : 0, gr = col_ok ? reflect101(x + 1, w) - x0 + 1 : 0;
  const int thr = (col_ok && thresh < 255) ? thresh : 0x7fffffff;
  const int rows = min(E2_TH, h - y0);
  int s0 = gray[0][gl] + gray[0][gr];
  int s1 = gray[1][gl] + gray[1][gr], c1 = gray[1][gc];
  const bool writer = lane == 0 && (x0 >> 5) + wq < words;
  const size_t o0 = (size_t(dst_slot) * h + y0) * words + (x0 >> 5) + wq;
  uint32_t* eo = edge_bits + o0;
  uint32_t* ro = REF ? ref_bits + o0 : nullptr;
  const D* dep = REF ? depth + sbase + size_t(y0) * w + (col_ok ? x : 0) : nullptr;
#pragma unroll 4
  for (int r = 0; r < rows; ++r) {
    const int s2 = gray[r + 2][gl] + gray[r + 2][gr], c2 = gray[r + 2][gc];
    const int v = 2 * (s0 + s2) - 8 * c1;
    const bool edge = abs(v) > thr;
    const unsigned eb = __ballot_sync(0xffffffffu, edge);
    if (REF) {
      bool valid = false;
      if (edge) valid = zero_to_one || dep[0] > D(0);
      const unsigned rb = __ballot_sync(0xffffffffu, valid);
      if (writer) *ro = rb;
      ro += words; dep += w;
    }
    if (writer) *eo = eb;
    eo += words;
    s0 = s1; s1 = s2; c1 = c2;
  }
}

// TW = tile width = threads per CTA (128; 64 for levels whose width is a multiple of 64 but not of 128, where a 128-wide
// last tile would be half empty).  REF: also write the reference-point plane (edge & depth > 0), key frames only.
// Instruction budget (the kernel is issue-bound, not HBM-bound): staging 6, blur + gray 31, Laplacian + ballot 12-16 per pixel.
template <typename D, int TW, bool REF>
__global__ void __launch_bounds__(TW) k_edge_mask2(const uint8_t* __restrict__ bgr, const D* __restrict__ depth,
                                                      size_t frame_stride_px, const int32_t* __restrict__ src_slots,
                                                      const int32_t* __restrict__ dst_slots, uint32_t* __restrict__ edge_bits,
                                                      uint32_t* __restrict__ ref_bits, int w, int h, int words, int thresh, int zero_to_one,
                                                      uint8_t* __restrict__ pyr_bgr, D* __restrict__ pyr_depth) {
  constexpr int PW = TW + 8;   // packed tile: image columns x0-4 .. x0+TW+3
  constexpr int GW = TW + 4;   // gray tile: columns x0-1 .. x0+TW (+2 pad)
  constexpr int NG = PW / 4;   // 4-pixel groups per tile row
  constexpr int RS = TW / NG;  // tile rows staged per pass (3)
  __shared__ unsigned tile[E2_PH][PW];
  __shared__ uint8_t gray[E2_TH + 2][GW];
  const int f = blockIdx.z;
  const size_t sbase = (src_slots ? size_t(src_slots[f]) : size_t(f)) * frame_stride_px;
  const int x0 = blockIdx.x * TW, y0 = blockIdx.y * E2_TH;
  const int t = threadIdx.x;
  const unsigned* img = reinterpret_cast<const unsigned*>(bgr + sbase * 3);
  const int row_words = (w * 3) >> 2;
  // ---- phase 1: 32-bit row loads, 3 words -> 4 packed pixels; a thread keeps its column group and walks down the rows ----
  {
    const int g = t % NG, rr = t / NG;
    const int col = x0 - 4 + 4 * g;                      // first image column of the group (multiple of 4)
    if (rr < RS && col >= 0 && col + 3 < w) {             // outside the image: never read (REFLECT_101 maps inside)
      const unsigned* src0 = img + (col * 3 >> 2);
#pragma unroll 2
      for (int r = rr; r < E2_PH; r += RS) {
        // rows y0-2 .. h+1 are all that the tile's outputs can reach (h >= 4: one reflection maps them inside); the rest stay unstaged
        const int y = y0 - 2 + r;
        if (y > h + 1) break;
        int ry = abs(y);
        ry = ry >= h ? 2 * h - 2 - ry : ry;
        const unsigned* src = src0 + size_t(unsigned(ry) * unsigned(row_words));
        const unsigned w0 = __ldg(src), w1 = __ldg(src + 1), w2 = __ldg(src + 2);
        uint4 px;
        px.x = w0 & 0x00FFFFFFu;
        px.y = __funnelshift_r(w0, w1, 24) & 0x00FFFFFFu;
        px.z = __funnelshift_r(w1, w2, 16) & 0x00FFFFFFu;
        px.w = w2 >> 8;
        *reinterpret_cast<uint4*>(&tile[r][4 * g]) = px;
      }
    }
  }
  __syncthreads();
  // ---- next pyramid level from the staged tile (pyr_bgr != null): cv::resize(0.5) INTER_LINEAR == 2x2 mean, (a+b+c+d+2) >> 2 per
  //      channel, four output pixels (12 bytes) per item; INTER_NEAREST on depth (key frames).  Saves a pass over the frame. ----
  if (pyr_bgr) {
    const int dw = w >> 1, dh = h >> 1;
    const size_t dbase = size_t(dst_slots[f]) * size_t(dw) * dh;
    for (int i = t; i < (TW / 8) * (E2_TH / 2); i += TW) {
      const int yl = i / (TW / 8), xq = i % (TW / 8);
      const int oy = (y0 >> 1) + yl, ox = (x0 >> 1) + 4 * xq;
      if (oy >= dh || ox + 3 >= dw) continue;
      const uint4 a0 = *reinterpret_cast<const uint4*>(&tile[2 * yl + 2][8 * xq + 4]), a1 = *reinterpret_cast<const uint4*>(&tile[2 * yl + 2][8 * xq + 8]);
      const uint4 b0 = *reinterpret_cast<const uint4*>(&tile[2 * yl + 3][8 * xq + 4]), b1 = *reinterpret_cast<const uint4*>(&tile[2 * yl + 3][8 * xq + 8]);
      const unsigned top[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w}, bot[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
      unsigned px[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        unsigned bg0, r0, bg1, r1, bg2, r2, bg3, r3;
        e2_expand(top[2 * j], bg0, r0); e2_expand(top[2 * j + 1], bg1, r1);
        e2_expand(bot[2 * j], bg2, r2); e2_expand(bot[2 * j + 1], bg3, r3);
        const unsigned sbg = ((bg0 + bg1 + bg2 + bg3 + 0x00020002u) >> 2) & 0x00FF00FFu;     // {B, G} means in 16-bit lanes
        const unsigned sr = (r0 + r1 + r2 + r3 + 2u) >> 2;
        px[j] = __byte_perm(sbg, sr, 0x4420);                                                // B | G << 8 | R << 16
      }
      unsigned* d = reinterpret_cast<unsigned*>(pyr_bgr + (dbase + size_t(oy) * dw + ox) * 3);
      d[0] = __byte_perm(px[0], px[1], 0x4210);
      d[1] = __byte_perm(px[1], px[2], 0x5421);
      d[2] = __byte_perm(px[2], px[3], 0x6542);
      if (REF && pyr_depth) {
        const D* sd = depth + sbase + size_t(2 * oy) * w + 2 * ox;
#pragma unroll
        for (int j = 0; j < 4; ++j) pyr_depth[dbase + size_t(oy) * dw + ox + j] = sd[2 * j];
      }
    }
  }
  // ---- phase 2: per-column rolling 3x3 blur + gray ----
  const int gx = x0 + t;
  if (gx < w) {
    const int cl = reflect101(gx - 1, w) - x0 + 4, cc = t + 4, cr = reflect101(gx + 1, w) - x0 + 4;
    unsigned hbg0 = 0, hr0 = 0, hbg1 = 0, hr1 = 0;
#pragma unroll 4
    for (int r = 0; r < E2_PH; ++r) {
      unsigned lbg, lr, cbg, crr, rbg, rr;
      e2_expand(tile[r][cl], lbg, lr);
      e2_expand(tile[r][cc], cbg, crr);
      e2_expand(tile[r][cr], rbg, rr);
      const unsigned hbg = lbg + rbg + (cbg << 1), hr = lr + rr + (crr << 1);
      if (r >= 2) gray[r - 2][t + 1] = uint8_t(e2_gray(hbg0 + hbg + (hbg1 << 1), hr0 + hr + (hr1 << 1)));
      hbg0 = hbg1; hr0 = hr1; hbg1 = hbg; hr1 = hr;
    }
  }
  // the two halo gray columns (x0-1 and x0+TW): 2 x 34 values, computed directly
  for (int q = t; q < 2 * (E2_TH + 2); q += TW) {
    const int which = q / (E2_TH + 2), gy = q % (E2_TH + 2);
    const int hx = which ? x0 + TW : x0 - 1;
    if (which == 0 || hx <= w) {                          // column w itself is still needed (reflect of w is w-2 ...)
      const int cl = reflect101(hx - 1, w) - x0 + 4, cc = reflect101(hx, w) - x0 + 4, cr = reflect101(hx + 1, w) - x0 + 4;
      if (cl >= 0 && cl < PW && cc >= 0 && cc < PW && cr >= 0 && cr < PW) {
        unsigned vbg = 0, vr = 0;
#pragma unroll
        for (int k = 0; k < 3; ++k) {
          unsigned lbg, lr, cbg, crr, rbg, rr;
          e2_expand(tile[gy + k][cl], lbg, lr);
          e2_expand(tile[gy + k][cc], cbg, crr);
          e2_expand(tile[gy + k][cr], rbg, rr);
          const unsigned m = (k == 1) ? 1u : 0u;
          vbg += (lbg + rbg + (cbg << 1)) << m;
          vr += (lr + rr + (crr << 1)) << m;
        }
        gray[gy][which ? TW + 1 : 0] = uint8_t(e2_gray(vbg, vr));
      }
    }
  }
  __syncthreads();
  // ---- phase 3 ----
  e2_laplacian_bits<D, TW, REF>(gray, depth, sbase, dst_slots[f], edge_bits, ref_bits, x0, y0, w, h, words, thresh, zero_to_one);
}

// ---- k_edge_mask2 on 8-bit gray input: the same edges as k_edge_mask2 on BGR (g, g, g), from a third of the bytes ----------
// RGB2GRAY of three equal blurred channels is the identity (9798 + 19235 + 3735 == 1 << 15, rounding constant half of it), so
// the blur goes straight into the gray tile.  The byte tile is staged REFLECT_101-padded (columns outside the image hold their
// mirror image), which makes every gray column -- the two halo columns too -- a contiguous 3-tap window: each thread blurs two
// adjacent columns in 16-bit lanes over one half of the tile's rows.  Phase 3 is k_edge_mask2's.  Needs w % 4 == 0.
// LUMA: where the luma bytes lie in the rows (img_pitch bytes apart; frames img_stride bytes apart; depth stays dense).
//   EA_LUMA_PLANAR  one byte per pixel (gray, the Y plane of NV12): 32-bit row loads, 4-byte aligned image, pitch and stride
//   EA_LUMA_YUYV    packed 4:2:2, Y at byte 2x (Y0 U Y1 V): one 8-byte load per 4 pixels, 8-byte aligned image, pitch, stride
//   EA_LUMA_UYVY    packed 4:2:2, Y at byte 2x + 1 (U Y0 V Y1): likewise
// Only phase 1 depends on it: the staged tile holds the same luma bytes in every layout.
enum { EA_LUMA_PLANAR = 0, EA_LUMA_YUYV = 1, EA_LUMA_UYVY = 2 };
template <typename D, int TW, bool REF, int LUMA>
__global__ void __launch_bounds__(TW) k_edge_mask2_gray(const uint8_t* __restrict__ src, size_t img_stride, unsigned img_pitch,
                                                          const D* __restrict__ depth,
                                                          size_t frame_stride_px, const int32_t* __restrict__ src_slots,
                                                          const int32_t* __restrict__ dst_slots, uint32_t* __restrict__ edge_bits,
                                                          uint32_t* __restrict__ ref_bits, int w, int h, int words, int thresh, int zero_to_one,
                                                          uint8_t* __restrict__ pyr, D* __restrict__ pyr_depth) {
  constexpr int PW = TW + 8;          // tile bytes per row: image columns x0-4 .. x0+TW+3
  constexpr int GW = TW + 4;          // gray tile: columns x0-1 .. x0+TW (+2 pad)
  constexpr int NG = PW / 4;          // 4-pixel words per tile row
  constexpr int RS = TW / NG;         // tile rows staged per pass
  constexpr int NP = (TW + 2) / 2;    // gray column pairs, halo columns included
  constexpr int H2 = (E2_TH + 2) / 2; // gray rows per half
  constexpr int STEP = LUMA == EA_LUMA_PLANAR ? 1 : 2, OFF = LUMA == EA_LUMA_UYVY ? 1 : 0;
  __shared__ __align__(16) uint8_t tile[E2_PH][PW];
  __shared__ __align__(16) uint8_t gray[E2_TH + 2][GW];
  const int f = blockIdx.z;
  const size_t sf = src_slots ? size_t(src_slots[f]) : size_t(f);
  const size_t sbase = sf * frame_stride_px;
  const int x0 = blockIdx.x * TW, y0 = blockIdx.y * E2_TH;
  const int t = threadIdx.x;
  const uint8_t* img = src + sf * img_stride;
  // ---- phase 1: one 32-bit (planar) or 64-bit (packed) load = 4 pixels; groups outside the image are gathered through
  //      REFLECT_101 byte by byte ----
  {
    const int g = t % NG, rr = t / NG;
    const int col = x0 - 4 + 4 * g;                       // first image column of the group (multiple of 4)
    const bool inside = col >= 0 && col + 3 < w;
    const int m0 = reflect101(col, w), m1 = reflect101(col + 1, w), m2 = reflect101(col + 2, w), m3 = reflect101(col + 3, w);
    if (rr < RS) {
#pragma unroll 2
      for (int r = rr; r < E2_PH; r += RS) {
        // rows y0-2 .. h+1 are all that the tile's outputs can reach (h >= 4: one reflection maps them inside); the rest stay unstaged
        const int y = y0 - 2 + r;
        if (y > h + 1) break;
        int ry = abs(y);
        ry = ry >= h ? 2 * h - 2 - ry : ry;
        const uint8_t* row = img + size_t(unsigned(ry)) * img_pitch;
        unsigned v;
        if (inside) {
          if constexpr (LUMA == EA_LUMA_PLANAR) {
            v = __ldg(reinterpret_cast<const unsigned*>(row + col));
          } else {
            const uint2 q = __ldg(reinterpret_cast<const uint2*>(row + 2 * col));
            v = __byte_perm(q.x, q.y, LUMA == EA_LUMA_YUYV ? 0x6420 : 0x7531);
          }
        } else {
          v = unsigned(row[STEP * m0 + OFF]) | unsigned(row[STEP * m1 + OFF]) << 8 | unsigned(row[STEP * m2 + OFF]) << 16 |
              unsigned(row[STEP * m3 + OFF]) << 24;
        }
        *reinterpret_cast<unsigned*>(&tile[r][4 * g]) = v;
      }
    }
  }
  __syncthreads();
  // ---- next pyramid level from the staged tile (pyr != null): (a+b+c+d+2) >> 2 in 16-bit lanes, four output pixels per 32-bit
  //      store; INTER_NEAREST on depth (key frames) ----
  if (pyr) {
    const int dw = w >> 1, dh = h >> 1;
    const size_t dbase = size_t(dst_slots[f]) * size_t(dw) * dh;
    for (int i = t; i < (TW / 8) * (E2_TH / 2); i += TW) {
      const int yl = i / (TW / 8), xq = i % (TW / 8);
      const int oy = (y0 >> 1) + yl, ox = (x0 >> 1) + 4 * xq;
      if (oy >= dh || ox + 3 >= dw) continue;
      const unsigned* a = reinterpret_cast<const unsigned*>(&tile[2 * yl + 2][8 * xq + 4]);
      const unsigned* b = reinterpret_cast<const unsigned*>(&tile[2 * yl + 3][8 * xq + 4]);
      // {p0 + p1, p2 + p3} of a 4-pixel word in 16-bit lanes
      auto pairs = [](unsigned v) { return __byte_perm(v, 0, 0x4240) + __byte_perm(v, 0, 0x4341); };
      const unsigned m01 = ((pairs(a[0]) + pairs(b[0]) + 0x00020002u) >> 2) & 0x00FF00FFu;
      const unsigned m23 = ((pairs(a[1]) + pairs(b[1]) + 0x00020002u) >> 2) & 0x00FF00FFu;
      *reinterpret_cast<unsigned*>(pyr + dbase + size_t(oy) * dw + ox) = __byte_perm(m01, m23, 0x6420);
      if (REF && pyr_depth) {
        const D* sd = depth + sbase + size_t(2 * oy) * w + 2 * ox;
#pragma unroll
        for (int j = 0; j < 4; ++j) pyr_depth[dbase + size_t(oy) * dw + ox + j] = sd[2 * j];
      }
    }
  }
  // ---- phase 2: rolling 3x3 blur of gray columns (g, g+1) <-> image columns x0-1+g, x0+g; item = (pair, half of the rows) ----
  for (int it = t; it < 2 * NP; it += TW) {
    const int g = 2 * (it % NP), r0 = (it / NP) * H2;
    const int wi = g >> 2;
    const bool aligned = (g & 2) != 0;                  // tile bytes g+2 .. g+5 (left, centre, centre, right) are word wi + 1
    unsigned h0 = 0, h1 = 0;
#pragma unroll 4
    for (int r = 0; r < H2 + 2; ++r) {
      const unsigned* row = reinterpret_cast<const unsigned*>(&tile[r0 + r][0]);
      const unsigned v = aligned ? row[wi + 1] : __byte_perm(row[wi], row[wi + 1], 0x5432);
      const unsigned hs = __byte_perm(v, 0, 0x4140) + (__byte_perm(v, 0, 0x4241) << 1) + __byte_perm(v, 0, 0x4342);
      if (r >= 2) {
        const unsigned s = ((h0 + hs + (h1 << 1) + 0x00080008u) >> 4) & 0x00FF00FFu;
        *reinterpret_cast<uint16_t*>(&gray[r0 + r - 2][g]) = uint16_t(__byte_perm(s, 0, 0x0020));
      }
      h0 = h1; h1 = hs;
    }
  }
  __syncthreads();
  // ---- phase 3 ----
  e2_laplacian_bits<D, TW, REF>(gray, depth, sbase, dst_slots[f], edge_bits, ref_bits, x0, y0, w, h, words, thresh, zero_to_one);
}

// ---- masks: keep set bits only where mask > thr (level l samples mask(x<<l, y<<l)) ----------------------------
//   reference points, get_aX_mask (utils.cpp:335,348): thr 0;  now-frame edges before the DT,
//   get_distance_transform2_masked[_NoNormalize] (utils.cpp:124-128,182-186: threshold(mask,1,1,BINARY)): thr 1
__global__ void __launch_bounds__(256) k_mask_ref_bits(uint32_t* __restrict__ ref_bits, const int32_t* __restrict__ dst_slots,
                                                       const uint8_t* __restrict__ mask, int w0, int h0, int w, int h, int words, int level,
                                                       int thr) {
  const int f = blockIdx.y;
  uint32_t* bits = ref_bits + size_t(dst_slots[f]) * h * words;
  const uint8_t* m = mask + size_t(f) * w0 * h0;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < h * words; i += gridDim.x * blockDim.x) {
    const int y = i / words, x0 = (i % words) * 32;
    unsigned keep = 0;
    unsigned b = bits[i];
    for (unsigned t = b; t; t &= t - 1) {
      const int k = __ffs(t) - 1;
      if (m[size_t(y << level) * w0 + ((x0 + k) << level)] > thr) keep |= 1u << k;
    }
    bits[i] = keep;
  }
}

// ---- ordered compaction: one CTA per frame, row-major rank == reference's loop order (utils.cpp:268-280) ----
#define CP_THREADS 1024
template <typename D>
__global__ void __launch_bounds__(CP_THREADS) k_compact(const uint32_t* __restrict__ ref_bits, const D* __restrict__ depth,
                                                        size_t frame_stride_px, const int32_t* __restrict__ src_slots,
                                                        const int32_t* __restrict__ dst_slots, float4* __restrict__ pts,
                                                        int* __restrict__ n_pts, int level, int* __restrict__ overflow,
                                                        int w, int h, int words, int cap, int zero_to_one, float depth_one,
                                                        const ea_track_info* __restrict__ gate) {
  __shared__ int warp_sums[CP_THREADS / 32];
  __shared__ int total_s;
  const int f = blockIdx.x;
  if (gate && gate[f].key_reasons == 0) return;                      // EA_COMPACT_ONLY: not promoted, no list needed
  const int slot = dst_slots[f];
  const uint32_t* bits = ref_bits + size_t(slot) * h * words;
  const D* dep = depth + (src_slots ? size_t(src_slots[f]) : size_t(f)) * frame_stride_px;
  uint2* out = reinterpret_cast<uint2*>(pts + size_t(slot) * cap);   // 8-byte pixel points at the head of the slot's 16 B x cap area
  const int nw = h * words;
  const int per = (nw + CP_THREADS - 1) / CP_THREADS;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int b = tid * per, e = min(b + per, nw);
  int cnt = 0;
  for (int i = b; i < e; ++i) cnt += __popc(bits[i]);
  int incl = cnt;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += t; }
  if (lane == 31) warp_sums[warp] = incl;
  __syncthreads();
  if (warp == 0) {
    int v = warp_sums[lane];
    int s = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, s, o); if (lane >= o) s += t; }
    warp_sums[lane] = s - v;
    if (lane == 31) total_s = s;
  }
  __syncthreads();
  int rank = warp_sums[warp] + incl - cnt;
  for (int i = b; i < e; ++i) {
    unsigned m = bits[i];
    const int y = i / words, xb = (i % words) * 32;
    while (m) {
      const int bit = __ffs(m) - 1;
      m &= m - 1;
      const int x = xb + bit;
      if (rank < cap) {
        float dz = float(dep[size_t(y) * w + x]);
        if (zero_to_one && dz == 0.0f) dz = depth_one;               // src/SolveEA.cpp:69
        out[rank] = ea_pack_pixel_point(unsigned(x), unsigned(y), dz);
      }
      ++rank;
    }
  }
  if (tid == 0) {
    n_pts[slot * EA_MAX_LEVELS + level] = min(total_s, cap);
    overflow[slot * EA_MAX_LEVELS + level] = total_s > cap ? 1 : 0;   // describes the list just written, not the frameset's history
  }
}

// ---- 3x3 median on the binary mask (cv::medianBlur(B,3), BORDER_REPLICATE), bit-parallel -------------------
// a, b, c: bit fields of rows y-1, y, y+1 where field bit p <-> pixel x0+p-1.  Returns the field of
// "at least 5 of the 9 neighbours are edge", bit k <-> pixel x0+k.
__device__ __forceinline__ unsigned long long median3_bits64(unsigned long long a, unsigned long long b, unsigned long long c) {
  const unsigned long long s0 = a ^ b ^ c, s1 = (a & b) | (c & (a ^ b));  // per-column vertical count = s0 + 2 s1
  const unsigned long long A0 = s0, B0 = s0 >> 1, C0 = s0 >> 2, A1 = s1, B1 = s1 >> 1, C1 = s1 >> 2;
  const unsigned long long lo = A0 ^ B0 ^ C0, carry = (A0 & B0) | (C0 & (A0 ^ B0));
  // m = A1 + B1 + C1 + carry ; total = lo + 2 m >= 5  <=>  m >= 3 or (m == 2 and lo)
  const unsigned long long t = A1 ^ B1, u = A1 & B1, v = C1 ^ carry, wv = C1 & carry;
  const unsigned long long m0 = t ^ v, tv = t & v;
  const unsigned long long ge1 = u | wv | tv, eq2 = u & wv;
  const unsigned long long m_ge3 = eq2 | (ge1 & m0);
  const unsigned long long m_eq2 = ge1 & ~eq2 & ~m0;
  return m_ge3 | (m_eq2 & lo);
}
__device__ __forceinline__ unsigned long long row_field64(const uint32_t* __restrict__ row, int wi, int words, int w) {
  const unsigned word = row[wi];
  const int nvalid = min(32, w - 32 * wi);
  const unsigned left = (wi > 0) ? (row[wi - 1] >> 31) : (word & 1u);
  unsigned right;
  if (nvalid == 32 && wi + 1 < words) right = row[wi + 1] & 1u;
  else right = (word >> (nvalid - 1)) & 1u;                         // replicate the last image column
  return (static_cast<unsigned long long>(word) << 1) | left | (static_cast<unsigned long long>(right) << (nvalid + 1));
}
__global__ void __launch_bounds__(256) k_median_bits(const __grid_constant__ EaPrepArgs A) {
  const int level = blockIdx.z;
  const EaPrepLevel& L = A.lv[level];
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= L.h * L.words) return;
  const int slot = A.slots[blockIdx.y];
  const uint32_t* bits = L.edge_bits + size_t(slot) * L.h * L.words;
  const int y = idx / L.words, wi = idx % L.words;
  const unsigned long long f0 = row_field64(bits + size_t(max(y - 1, 0)) * L.words, wi, L.words, L.w);
  const unsigned long long f1 = row_field64(bits + size_t(y) * L.words, wi, L.words, L.w);
  const unsigned long long f2 = row_field64(bits + size_t(min(y + 1, L.h - 1)) * L.words, wi, L.words, L.w);
  const int nvalid = min(32, L.w - 32 * wi);
  unsigned m = unsigned(median3_bits64(f0, f1, f2));
  if (nvalid < 32) m &= (1u << nvalid) - 1u;
  L.med_bits[size_t(slot) * L.h * L.words + idx] = m;
}

// ---- chamfer 3x3 distance transform, OpenCV's fixed-point two-pass recurrence (distanceTransform_3x3) -------
// One CTA per (frame, level); rows are sequential, each row is a block-wide min-plus scan (thread-local P
// pixels -> warp shuffle scan -> cross-warp carry through shared memory, ONE barrier per row).  Integer min/+
// is associative, so the scan reproduces the raster recurrence bit for bit.  The previous row lives in
// registers; only warp totals / boundary pixels go through shared memory (parity double-buffered).
#define DT_HV 62587         // cvRound(0.955f  * 65536)
#define DT_DG 89738         // cvRound(1.3693f * 65536)
#define DT_INF 0x3FFFFFFF   // internal "no seed yet"; written out as OpenCV's DIST_MAX
#define DT_DISTMAX (0xFFFFFFFFu - 89738u)

template <int P, bool BACKWARD>
__device__ __forceinline__ void dt_row_scan(int (&d)[P], const int (&cval)[P], int lane, int warp, int n_warps, int par,
                                            int (*tot)[32], int (*first)[32], int& left_bnd, int& right_bnd) {
  // local scan inside the thread (scan direction: increasing k for the forward pass, decreasing for the backward)
  int dl[P];
  int run = DT_INF;
#pragma unroll
  for (int kk = 0; kk < P; ++kk) {
    const int k = BACKWARD ? (P - 1 - kk) : kk;
    run = min(cval[k], run + DT_HV);
    dl[k] = run;
  }
  // warp scan of the thread totals; "upstream" = lower lanes (forward) / higher lanes (backward)
  const int pos = BACKWARD ? (31 - lane) : lane;   // position along the scan direction
  const int stepP = DT_HV * P;
  int e = min(run, DT_INF) - stepP * pos;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int t = BACKWARD ? __shfl_down_sync(0xffffffffu, e, o) : __shfl_up_sync(0xffffffffu, e, o);
    if (pos >= o) e = min(e, t);
  }
  const int out = e + stepP * pos;                 // value of this thread's last pixel, ignoring the block carry
  int carry_local = BACKWARD ? __shfl_down_sync(0xffffffffu, out, 1) : __shfl_up_sync(0xffffffffu, out, 1);
  if (pos == 0) carry_local = DT_INF;
  const int Lw = __shfl_sync(0xffffffffu, out, BACKWARD ? 0 : 31);
  const int f0 = __shfl_sync(0xffffffffu, BACKWARD ? dl[P - 1] : dl[0], BACKWARD ? 31 : 0);
  if (lane == 0) { tot[par][warp] = min(Lw, DT_INF); first[par][warp] = min(f0, DT_INF); }
  __syncthreads();
  // block carry: final value of the pixel just upstream of this warp
  const int wpos = BACKWARD ? (n_warps - 1 - warp) : warp;
  const int stepW = stepP * 32;
  int cand = DT_INF;
  if (lane < wpos) {
    const int src = BACKWARD ? (n_warps - 1 - lane) : lane;
    cand = tot[par][src] + stepW * (wpos - 1 - lane);
  }
  const int cw = min(__reduce_min_sync(0xffffffffu, cand), DT_INF);
#pragma unroll
  for (int kk = 0; kk < P; ++kk) {
    const int k = BACKWARD ? (P - 1 - kk) : kk;
    const int v = min(min(dl[k], carry_local + DT_HV * (kk + 1)), cw + DT_HV * (pos * P + kk + 1));
    d[k] = min(v, DT_INF);
  }
  // boundaries the NEXT row needs: upstream neighbour's last pixel (== cw) and downstream neighbour's first pixel
  const int out_w = min(min(Lw, cw + stepW), DT_INF);
  const int dn = BACKWARD ? warp - 1 : warp + 1;
  const int dn_first = (dn >= 0 && dn < n_warps) ? min(first[par][dn], out_w + DT_HV) : DT_INF;
  if (BACKWARD) { right_bnd = cw; left_bnd = dn_first; }
  else { left_bnd = cw; right_bnd = dn_first; }
}

// P consecutive 32-bit values of one row: 128-bit accesses when the row layout allows it (w % 4 == 0, P % 4 == 0)
template <int P, typename T>
__device__ __forceinline__ void dt_store_row(T* __restrict__ row, int x0, int w, const T (&v)[P], bool vec_ok) {
  if (vec_ok && x0 + P <= w) {
#pragma unroll
    for (int k = 0; k < P; k += 4) *reinterpret_cast<int4*>(row + x0 + k) = *reinterpret_cast<const int4*>(&v[k]);
  } else {
#pragma unroll
    for (int k = 0; k < P; ++k) if (x0 + k < w) row[x0 + k] = v[k];
  }
}
template <int P>
__device__ __forceinline__ void dt_load_row(const int* __restrict__ row, int x0, int w, int (&v)[P], bool vec_ok) {
  if (vec_ok && x0 + P <= w) {
#pragma unroll
    for (int k = 0; k < P; k += 4) *reinterpret_cast<int4*>(&v[k]) = *reinterpret_cast<const int4*>(row + x0 + k);
  } else {
#pragma unroll
    for (int k = 0; k < P; ++k) v[k] = (x0 + k < w) ? row[x0 + k] : DT_INF;
  }
}

template <int P>
__global__ void __launch_bounds__(1024) k_chamfer_dt(const __grid_constant__ EaPrepArgs A) {
  __shared__ int tot[2][32], first[2][32];
  __shared__ unsigned red[2][32];
  const int level = blockIdx.y;
  const EaPrepLevel& L = A.lv[level];
  const int w = L.w, h = L.h, words = L.words;
  const int slot = A.slots[blockIdx.x];
  const uint32_t* bits = (A.use_median ? L.med_bits : L.edge_bits) + size_t(slot) * h * words;
  float* gf = ea_dt_origin(L, slot);                 // pixel (0,0) of the padded image; rows are pitch apart
  int* gi = reinterpret_cast<int*>(gf);
  const int pitch = L.dt_pitch;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int n_warps = ((w + P - 1) / P + 31) / 32;          // warps that own pixels at this level
  const bool warp_on = warp < n_warps;
  const int x0 = tid * P;
  const bool vec_ok = (P % 4 == 0) && ((w & 3) == 0);
  int d[P];
#pragma unroll
  for (int k = 0; k < P; ++k) d[k] = DT_INF;
  int left_bnd = DT_INF, right_bnd = DT_INF;
  int par = 0;
  // ---------------- forward pass: rows top -> bottom, scan left -> right ----------------
  unsigned ebits_next = (warp_on && x0 < w) ? bits[x0 >> 5] : 0u;
  for (int y = 0; y < h; ++y, par ^= 1) {
    if (!warp_on) { __syncthreads(); continue; }
    const unsigned ebits = ebits_next >> (x0 & 31);
    if (x0 < w && y + 1 < h) ebits_next = bits[size_t(y + 1) * words + (x0 >> 5)];   // prefetch the next row's mask word
    int pl = __shfl_up_sync(0xffffffffu, d[P - 1], 1);
    int pr = __shfl_down_sync(0xffffffffu, d[0], 1);
    if (lane == 0) pl = left_bnd;
    if (lane == 31) pr = right_bnd;
    int cval[P];
#pragma unroll
    for (int k = 0; k < P; ++k) {
      const int a = (k == 0) ? pl : d[k - 1];
      const int c = (k == P - 1) ? pr : d[k + 1];
      int v = min(min(a, c) + DT_DG, d[k] + DT_HV);
      if ((ebits >> k) & 1u) v = 0;
      if (x0 + k >= w) v = DT_INF;                           // beyond the image: stays "border"
      cval[k] = min(v, DT_INF);
    }
    dt_row_scan<P, false>(d, cval, lane, warp, n_warps, par, tot, first, left_bnd, right_bnd);
#pragma unroll
    for (int k = 0; k < P; ++k) if (x0 + k >= w) d[k] = DT_INF;
    if (x0 < w) dt_store_row<P, int>(gi + size_t(y) * pitch, x0, w, d, vec_ok);
  }
  // ---------------- backward pass: rows bottom -> top, scan right -> left ----------------
#pragma unroll
  for (int k = 0; k < P; ++k) d[k] = DT_INF;
  left_bnd = DT_INF; right_bnd = DT_INF;
  unsigned vmax = 0, vmin = 0xFFFFFFFFu;
  int t_next[P];
#pragma unroll
  for (int k = 0; k < P; ++k) t_next[k] = DT_INF;
  if (warp_on && x0 < w) dt_load_row<P>(gi + size_t(h - 1) * pitch, x0, w, t_next, vec_ok);
  for (int y = h - 1; y >= 0; --y, par ^= 1) {
    if (!warp_on) { __syncthreads(); continue; }
    int t0[P];
#pragma unroll
    for (int k = 0; k < P; ++k) t0[k] = t_next[k];
    if (y > 0 && x0 < w) dt_load_row<P>(gi + size_t(y - 1) * pitch, x0, w, t_next, vec_ok);   // prefetch the next row up
    int pl = __shfl_up_sync(0xffffffffu, d[P - 1], 1);
    int pr = __shfl_down_sync(0xffffffffu, d[0], 1);
    if (lane == 0) pl = left_bnd;
    if (lane == 31) pr = right_bnd;
    int cval[P];
#pragma unroll
    for (int k = 0; k < P; ++k) {
      const int a = (k == 0) ? pl : d[k - 1];
      const int c = (k == P - 1) ? pr : d[k + 1];
      int v = min(t0[k], min(min(a, c) + DT_DG, d[k] + DT_HV));
      if (x0 + k >= w) v = DT_INF;
      cval[k] = min(v, DT_INF);
    }
    dt_row_scan<P, true>(d, cval, lane, warp, n_warps, par, tot, first, left_bnd, right_bnd);
    float outv[P];
#pragma unroll
    for (int k = 0; k < P; ++k) {
      outv[k] = 0.0f;
      if (x0 + k >= w) { d[k] = DT_INF; continue; }
      const unsigned t = (d[k] >= DT_INF) ? DT_DISTMAX : unsigned(d[k]);
      vmax = max(vmax, t); vmin = min(vmin, t);
      outv[k] = float(t) * (1.0f / 65536.0f);
    }
    if (x0 < w) dt_store_row<P, float>(gf + size_t(y) * pitch, x0, w, outv, vec_ok);
  }
  vmax = __reduce_max_sync(0xffffffffu, vmax);
  vmin = __reduce_min_sync(0xffffffffu, vmin);
  if (lane == 0) { red[0][warp] = vmin; red[1][warp] = vmax; }
  __syncthreads();
  if (tid == 0) {
    unsigned mn = 0xFFFFFFFFu, mx = 0;
    for (int i = 0; i < n_warps; ++i) { mn = min(mn, red[0][i]); mx = max(mx, red[1][i]); }
    A.dt_minmax[(slot * EA_MAX_LEVELS + level) * 2] = mn;
    A.dt_minmax[(slot * EA_MAX_LEVELS + level) * 2 + 1] = mx;
    // cv::normalize(NORM_MINMAX, alpha = 0, beta): scale = beta / (max - min), shift = -min * scale (double, then float)
    float2 aff = make_float2(1.0f, 0.0f);
    if (A.dt_normalize != EA_NORM_NONE) {
      const double beta = (A.dt_normalize == EA_NORM_255) ? 255.0 : 1.0;
      const float fmn = float(mn) * (1.0f / 65536.0f), fmx = float(mx) * (1.0f / 65536.0f);
      const double range = double(fmx) - double(fmn);
      const double scale = beta * (range > 2.220446049250313e-16 ? 1.0 / range : 0.0);
      aff = make_float2(float(scale), float(0.0 - double(fmn) * scale));
    }
    A.dt_affine[slot * EA_MAX_LEVELS + level] = aff;
  }
}

// ---- chamfer 3x3 DT, one WARP per (frame, level) ---------------------------------------------------------------------
// Same recurrence and results as k_chamfer_dt.  Each lane owns a contiguous strip of P pixels of the row, so the
// horizontal min-plus scan is P register steps plus ONE 5-step warp scan per row: no shared memory, no block barrier, and
// the per-row overhead is spread over P = 20 pixels at 640 px instead of 4 (the block kernel spends most of its
// instructions on scan / carry plumbing).  592 frames x 3 levels = 1 776 independent warps keep every scheduler busy
// without any of them waiting for another.  Used when every level is at most 32 * DTW_PMAX pixels wide.
#define DTW_PMAX 20
template <int P, bool BACKWARD, int SEG>
__device__ __forceinline__ void dtw_row_scan(int (&d)[P], const int (&cval)[P], const int lp) {   // lp: lane within its segment
  // A single warp per scheduler cannot hide latency with other warps, so the row step is arranged for short dependency
  // chains: with the ramp HV * position taken out, the strip total is a tree minimum (feeds the warp scan at once) and the
  // strip-local prefix minimum is a two-level scan that overlaps the shuffles.
  static_assert(P % 4 == 0, "strip length must be a multiple of 4");
  int e[P];                         // e[kk] = value at scan position kk minus HV * kk
#pragma unroll
  for (int kk = 0; kk < P; ++kk) e[kk] = cval[BACKWARD ? (P - 1 - kk) : kk] - DT_HV * kk;
  int m[P / 4];
#pragma unroll
  for (int g = 0; g < P / 4; ++g) m[g] = min(min(e[4 * g], e[4 * g + 1]), min(e[4 * g + 2], e[4 * g + 3]));
  int mt = m[0];
#pragma unroll
  for (int g = 1; g < P / 4; ++g) mt = min(mt, m[g]);
  const int run = min(mt + DT_HV * (P - 1), DT_INF);          // the strip's last pixel, ignoring upstream strips
  const int pos = BACKWARD ? (SEG - 1 - lp) : lp;
  constexpr int stepP = DT_HV * P;
  int s = run - stepP * pos;
#pragma unroll
  for (int o = 1; o < SEG; o <<= 1) {
    const int t = BACKWARD ? __shfl_down_sync(0xffffffffu, s, o, SEG) : __shfl_up_sync(0xffffffffu, s, o, SEG);
    if (pos >= o) s = min(s, t);
  }
  const int out = s + stepP * pos;   // final value of this lane's last pixel along the scan
  int carry = BACKWARD ? __shfl_down_sync(0xffffffffu, out, 1, SEG) : __shfl_up_sync(0xffffffffu, out, 1, SEG);
  if (pos == 0) carry = DT_INF;
  carry = min(carry, DT_INF);
  // strip-local prefix minimum (independent of the shuffles above)
  int gp[P / 4];                    // minimum of all groups before g
  gp[0] = DT_INF;
#pragma unroll
  for (int g = 1; g < P / 4; ++g) gp[g] = min(gp[g - 1], m[g - 1]);
#pragma unroll
  for (int g = 0; g < P / 4; ++g) {
    int pm = gp[g];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int kk = 4 * g + i;
      pm = min(pm, e[kk]);
      const int v = min(pm, carry + DT_HV) + DT_HV * kk;                 // min(local, carry + HV * (kk + 1)); >= DT_INF means no seed yet
      d[BACKWARD ? (P - 1 - kk) : kk] = v;
    }
  }
}

// FULL: every lane's strip lies inside the image (w == 32 * P, e.g. 640 px at P = 20): the per-pixel bound checks drop out.
#define DTW_L2_AHEAD 4      // rows of L2 prefetch distance (measured: see profiles)
// SEG: lanes per frame.  A row of 32 * P pixels takes the whole warp; the coarser pyramid levels of a 640-pixel frame (320, 160,
// 80 pixels) would leave most strips empty -- and paid 2-3x the instructions per pixel of level 0 -- so they run as 2 / 4 / 8
// frames side by side in one warp, each on SEG = 16 / 8 / 4 lanes with the same full 20-pixel strips (segmented shuffles).
template <int P, bool FULL, int SEG>
__device__ __forceinline__ void dtw_level(const EaPrepArgs& A, const int level, const int lane) {
  const EaPrepLevel& L = A.lv[level];
  const int lp = lane % SEG;                                       // lane within the frame's segment
  const int fi = int(blockIdx.x) * (32 / SEG) + lane / SEG;        // frame of this segment
  const bool frame_on = fi < A.n;
  const int slot = A.slots[frame_on ? fi : 0];
  const unsigned seg_mask = (0xffffffffu >> (32 - SEG)) << ((lane / SEG) * SEG);
  const int w = FULL ? SEG * P : L.w, h = L.h, words = L.words;   // FULL: a compile-time width folds every bound check
  const uint32_t* bits = (A.use_median ? L.med_bits : L.edge_bits) + size_t(slot) * h * words;
  float* gf = ea_dt_origin(L, slot);                 // pixel (0,0) of the padded image; rows are pitch apart
  int* gi = reinterpret_cast<int*>(gf);
  const int pitch = L.dt_pitch;
  const int x0 = lp * P;
  const bool on = frame_on && x0 < w;
  const bool vec_ok = (P % 4 == 0) && ((w & 3) == 0);
  const int wi = x0 >> 5, sh = x0 & 31;
  const bool two = on && (wi + 1 < words);
  int d[P];
#pragma unroll
  for (int k = 0; k < P; ++k) d[k] = DT_INF;
  // ---------------- forward pass ----------------
  unsigned b0 = on ? bits[wi] : 0u, b1 = two ? bits[wi + 1] : 0u;
  for (int y = 0; y < h; ++y) {
    const unsigned ebits = __funnelshift_r(b0, b1, sh);
    if (y + DTW_L2_AHEAD < h && lp == 0) asm volatile("prefetch.global.L2 [%0];" ::"l"(bits + size_t(y + DTW_L2_AHEAD) * words));
    if (y + 1 < h) {   // prefetch the next row's mask words
      b0 = on ? bits[size_t(y + 1) * words + wi] : 0u;
      b1 = two ? bits[size_t(y + 1) * words + wi + 1] : 0u;
    }
    int pl = __shfl_up_sync(0xffffffffu, d[P - 1], 1, SEG);
    int pr = __shfl_down_sync(0xffffffffu, d[0], 1, SEG);
    if (lp == 0) pl = DT_INF;
    if (lp == SEG - 1) pr = DT_INF;
    int cval[P];
#pragma unroll
    for (int k = 0; k < P; ++k) {
      const int a = (k == 0) ? pl : d[k - 1];
      const int c = (k == P - 1) ? pr : d[k + 1];
      int v = min(min(a, c) + DT_DG, d[k] + DT_HV);
      if ((ebits >> k) & 1u) v = 0;
      if (!FULL && x0 + k >= w) v = DT_INF;
      cval[k] = v;     // "infinite" values stay >= DT_INF and bounded by DT_INF + DG + HV * P (the carry below is clamped every row)
    }
    dtw_row_scan<P, false, SEG>(d, cval, lp);
#pragma unroll
    for (int k = 0; k < P; ++k) if (!FULL && x0 + k >= w) d[k] = DT_INF;
    if (on) dt_store_row<P, int>(gi + size_t(y) * pitch, x0, w, d, vec_ok);
  }
  // ---------------- backward pass ----------------
#pragma unroll
  for (int k = 0; k < P; ++k) d[k] = DT_INF;
  unsigned vmax = 0, vmin = 0xFFFFFFFFu;
  int t_next[P];
#pragma unroll
  for (int k = 0; k < P; ++k) t_next[k] = DT_INF;
  __syncwarp();   // the forward rows were written by other lanes' neighbours only through registers; own rows are re-read below
  if (on) dt_load_row<P>(gi + size_t(h - 1) * pitch, x0, w, t_next, vec_ok);
  for (int y = h - 1; y >= 0; --y) {
    int t0[P];
#pragma unroll
    for (int k = 0; k < P; ++k) t0[k] = t_next[k];
    if (y > 0 && on) dt_load_row<P>(gi + size_t(y - 1) * pitch, x0, w, t_next, vec_ok);
    // the forward rows were written ~1 ms ago and have left the L2: the register prefetch one row ahead does not cover a
    // DRAM round trip (ncu: 31 % of the kernel's samples waited here), so rows further up are pulled into L2 early
    if (y >= DTW_L2_AHEAD && frame_on && lp * 32 < w)
      asm volatile("prefetch.global.L2 [%0];" ::"l"(gi + size_t(y - DTW_L2_AHEAD) * pitch + lp * 32));
    int pl = __shfl_up_sync(0xffffffffu, d[P - 1], 1, SEG);
    int pr = __shfl_down_sync(0xffffffffu, d[0], 1, SEG);
    if (lp == 0) pl = DT_INF;
    if (lp == SEG - 1) pr = DT_INF;
    int cval[P];
#pragma unroll
    for (int k = 0; k < P; ++k) {
      const int a = (k == 0) ? pl : d[k - 1];
      const int c = (k == P - 1) ? pr : d[k + 1];
      int v = min(t0[k], min(min(a, c) + DT_DG, d[k] + DT_HV));
      if (!FULL && x0 + k >= w) v = DT_INF;
      cval[k] = v;     // "infinite" values stay >= DT_INF and bounded by DT_INF + DG + HV * P (the carry below is clamped every row)
    }
    dtw_row_scan<P, true, SEG>(d, cval, lp);
    float outv[P];
#pragma unroll
    for (int k = 0; k < P; ++k) {
      outv[k] = 0.0f;
      if (!FULL && x0 + k >= w) { d[k] = DT_INF; continue; }
      const unsigned t = (d[k] >= DT_INF) ? DT_DISTMAX : unsigned(d[k]);
      vmax = max(vmax, t); vmin = min(vmin, t);
      outv[k] = float(t) * (1.0f / 65536.0f);
    }
    // the finished row plus its share of the replicated border (EA_DT_PAD): the left / right 4 columns, and the 4 rows
    // above the first / below the last image row
    const int copies = (y == 0 || y == h - 1) ? 1 + EA_DT_PAD : 1;
    const int ystep = (y == 0) ? -1 : 1;
    const bool last_strip = on && (x0 + P >= w);
    float edge_r = 0.0f;
    if (last_strip) {
#pragma unroll
      for (int k = 0; k < P; ++k) if (x0 + k == w - 1) edge_r = outv[k];
    }
    for (int c = 0; c < copies; ++c) {
      float* row = gf + (ptrdiff_t(y) + ptrdiff_t(c) * ystep) * pitch;
      if (on) dt_store_row<P, float>(row, x0, w, outv, vec_ok);
      if (lp == 0 && frame_on) *reinterpret_cast<float4*>(row - EA_DT_PAD) = make_float4(outv[0], outv[0], outv[0], outv[0]);
      if (last_strip) for (int x = w; x < pitch - EA_DT_PAD; ++x) row[x] = edge_r;
    }
    if (h == 1 && y == 0) {   // a single image row is both first and last: the rows below it as well
      for (int c = 1; c <= EA_DT_PAD; ++c) {
        float* row = gf + ptrdiff_t(c) * pitch;
        if (on) dt_store_row<P, float>(row, x0, w, outv, vec_ok);
        if (lp == 0 && frame_on) *reinterpret_cast<float4*>(row - EA_DT_PAD) = make_float4(outv[0], outv[0], outv[0], outv[0]);
        if (last_strip) for (int x = w; x < pitch - EA_DT_PAD; ++x) row[x] = edge_r;
      }
    }
  }
  const unsigned mx = __reduce_max_sync(seg_mask, vmax);
  const unsigned mn = __reduce_min_sync(seg_mask, vmin);
  if (lp == 0 && frame_on) {
    A.dt_minmax[(slot * EA_MAX_LEVELS + level) * 2] = mn;
    A.dt_minmax[(slot * EA_MAX_LEVELS + level) * 2 + 1] = mx;
    // cv::normalize(NORM_MINMAX, alpha = 0, beta): scale = beta / (max - min), shift = -min * scale (double, then float)
    float2 aff = make_float2(1.0f, 0.0f);
    if (A.dt_normalize != EA_NORM_NONE) {
      const double beta = (A.dt_normalize == EA_NORM_255) ? 255.0 : 1.0;
      const float fmn = float(mn) * (1.0f / 65536.0f), fmx = float(mx) * (1.0f / 65536.0f);
      const double range = double(fmx) - double(fmn);
      const double scale = beta * (range > 2.220446049250313e-16 ? 1.0 / range : 0.0);
      aff = make_float2(float(scale), float(0.0 - double(fmn) * scale));
    }
    A.dt_affine[slot * EA_MAX_LEVELS + level] = aff;
  }
}

// lanes per frame at a level of width w: full 20-pixel strips on 16 / 8 / 4 lanes where the width allows it, else the whole warp
__host__ __device__ __forceinline__ int dtw_seg(int w) {
  return w == 16 * DTW_PMAX ? 16 : w == 8 * DTW_PMAX ? 8 : w == 4 * DTW_PMAX ? 4 : 32;
}
__global__ void __launch_bounds__(32) k_chamfer_dt_warp(const __grid_constant__ EaPrepArgs A) {
  const int level = blockIdx.y, lane = threadIdx.x;
  const int w = A.lv[level].w;
  const int seg = dtw_seg(w);
  if (int(blockIdx.x) * (32 / seg) >= A.n) return;           // the grid is sized for one frame per warp (level 0)
  const int per = (w + 31) / 32;
  if (seg == 16) dtw_level<DTW_PMAX, true, 16>(A, level, lane);
  else if (seg == 8) dtw_level<DTW_PMAX, true, 8>(A, level, lane);
  else if (seg == 4) dtw_level<DTW_PMAX, true, 4>(A, level, lane);
  else if (per <= 8) { if (w == 256) dtw_level<8, true, 32>(A, level, lane); else dtw_level<8, false, 32>(A, level, lane); }
  else if (per <= 12) { if (w == 384) dtw_level<12, true, 32>(A, level, lane); else dtw_level<12, false, 32>(A, level, lane); }
  else { if (w == 32 * DTW_PMAX) dtw_level<DTW_PMAX, true, 32>(A, level, lane); else dtw_level<DTW_PMAX, false, 32>(A, level, lane); }
}

// ---- normalised copy of one DT (read-back for parity tests): dst = raw * scale + shift, exactly as cv::normalize ----
__global__ void __launch_bounds__(256) k_dt_normalized_copy(const float* __restrict__ origin, int pitch, const float2* __restrict__ affine,
                                                            int w, int h, float* __restrict__ out) {
  const float2 a = *affine;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < w * h; i += gridDim.x * blockDim.x)
    out[i] = __fadd_rn(__fmul_rn(origin[size_t(i / w) * pitch + (i % w)], a.x), a.y);
}

// ---- padded layout helpers (EA_DT_PAD): every element of the padded image = the nearest image pixel --------------------
// import: from a dense [h][w] source (ea_frameset_set_dt);  fill_pad: border only, from the interior already in place
__global__ void __launch_bounds__(256) k_dt_import(const float* __restrict__ src, float* __restrict__ origin, int w, int h, int pitch) {
  const int n = pitch * (h + 2 * EA_DT_PAD);
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const int py = i / pitch - EA_DT_PAD, px = i % pitch - EA_DT_PAD;
    origin[ptrdiff_t(py) * pitch + px] = src[size_t(min(max(py, 0), h - 1)) * w + min(max(px, 0), w - 1)];
  }
}
__global__ void __launch_bounds__(256) k_dt_fill_pad(float* __restrict__ pool, size_t slot_floats, const int32_t* __restrict__ slots,
                                                     int w, int h, int pitch) {
  float* origin = pool + size_t(slots[blockIdx.y]) * slot_floats + size_t(EA_DT_PAD) * pitch + EA_DT_PAD;
  const int n = pitch * (h + 2 * EA_DT_PAD);
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const int py = i / pitch - EA_DT_PAD, px = i % pitch - EA_DT_PAD;
    if (py >= 0 && py < h && px >= 0 && px < w) continue;
    origin[ptrdiff_t(py) * pitch + px] = origin[size_t(min(max(py, 0), h - 1)) * pitch + min(max(px, 0), w - 1)];
  }
}

__global__ void __launch_bounds__(256) k_unpack_mask(const uint32_t* __restrict__ bits, int w, int h, int words, int median,
                                                     uint8_t* __restrict__ out) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < w * h; i += gridDim.x * blockDim.x) {
    const int x = i % w, y = i / w;
    int edge;
    if (!median) edge = (bits[size_t(y) * words + (x >> 5)] >> (x & 31)) & 1;
    else {
      int cnt = 0;
      for (int dy = -1; dy <= 1; ++dy)
        for (int dx = -1; dx <= 1; ++dx) {
          const int xx = min(max(x + dx, 0), w - 1), yy = min(max(y + dy, 0), h - 1);
          cnt += (bits[size_t(yy) * words + (xx >> 5)] >> (xx & 31)) & 1;
        }
      edge = cnt >= 5;
    }
    out[i] = edge ? 0 : 255;   // reference convention: B == 0 on edges (utils.cpp:60-70)
  }
}

}  // namespace

// the gray edge kernel loads whole 32-bit words (planar) or 64-bit words (packed 4:2:2) of level l's image: a caller's image whose
// address, row pitch or frame stride is not 4- / 8-byte aligned takes the byte path (k_edge_mask) instead
static bool gray_words_ok(const EaPrepArgs& A, int l) {
  if (A.in_format == EA_IMAGE_BGR8) return true;
  const EaImage m = ea_level_image(A, l);
  const uintptr_t align = m.step == 1 ? 3 : 7;
  return ((reinterpret_cast<uintptr_t>(m.base) | m.stride | m.pitch) & align) == 0;
}
// can level l's Laplacian edge kernel (k_edge_mask2 / k_edge_mask2_gray) also emit level l + 1's image / depth from its staged
// tile?  (Both store whole 32-bit words of level l + 1: 4 BGR pixels in 3 words, or 4 gray pixels in one; next level's width a
// multiple of 4 and a 4-byte aligned pool keep every such word aligned in either layout.)
static bool edge_kernel_fuses_pyramid(const EaPrepArgs& A, int l) {
  if (l + 1 >= A.n_levels || A.edge_detector != EA_EDGE_LAPLACIAN) return false;
  const EaPrepLevel& L = A.lv[l];
  const EaPrepLevel& N = A.lv[l + 1];
  return (L.w & 3) == 0 && L.w >= 8 && L.h >= 4 && gray_words_ok(A, l) && (N.w & 3) == 0 && (reinterpret_cast<uintptr_t>(N.bgr) & 3) == 0;
}

// the fused edge kernel of one level (k_edge_mask2 on BGR, k_edge_mask2_gray in the luma layout of one-channel input)
template <typename D, int TW, bool REF>
static void launch_edge_mask2(const EaPrepArgs& A, const EaPrepLevel& L, const EaImage& m, const D* d, size_t pxl, const int32_t* ss,
                              uint8_t* nb, D* nd, cudaStream_t stream) {
  dim3 grid(unsigned((L.w + TW - 1) / TW), unsigned((L.h + E2_TH - 1) / E2_TH), unsigned(A.n));
  uint32_t* rb = REF ? L.ref_bits : nullptr;
  const unsigned pitch = unsigned(m.pitch);
  if (A.in_format == EA_IMAGE_BGR8)
    k_edge_mask2<D, TW, REF><<<grid, TW, 0, stream>>>(m.base, d, pxl, ss, A.slots, L.edge_bits, rb, L.w, L.h, L.words, A.grad_threshold, A.zero_to_one, nb, nd);
  else if (m.step == 1)
    k_edge_mask2_gray<D, TW, REF, EA_LUMA_PLANAR><<<grid, TW, 0, stream>>>(m.base, m.stride, pitch, d, pxl, ss, A.slots, L.edge_bits, rb, L.w, L.h, L.words, A.grad_threshold, A.zero_to_one, nb, nd);
  else if (m.offset == 0)
    k_edge_mask2_gray<D, TW, REF, EA_LUMA_YUYV><<<grid, TW, 0, stream>>>(m.base, m.stride, pitch, d, pxl, ss, A.slots, L.edge_bits, rb, L.w, L.h, L.words, A.grad_threshold, A.zero_to_one, nb, nd);
  else
    k_edge_mask2_gray<D, TW, REF, EA_LUMA_UYVY><<<grid, TW, 0, stream>>>(m.base, m.stride, pitch, d, pxl, ss, A.slots, L.edge_bits, rb, L.w, L.h, L.words, A.grad_threshold, A.zero_to_one, nb, nd);
}

// the point lists of one level from the ref_bits plane and the depth (level 0: the caller's input by frame; above: the slot's pyramid)
template <typename D>
static void launch_compact(const EaPrepArgs& A, int l, cudaStream_t stream) {
  const EaPrepLevel& L = A.lv[l];
  const D* d = (l == 0) ? static_cast<const D*>(A.in_depth) : static_cast<const D*>(L.depth);
  k_compact<D><<<A.n, CP_THREADS, 0, stream>>>(L.ref_bits, d, size_t(L.w) * L.h, (l == 0) ? nullptr : A.slots, A.slots, L.pts, A.n_pts, l,
                                               A.overflow, L.w, L.h, L.words, L.cap, A.zero_to_one, A.depth_one,
                                               A.compact == EA_COMPACT_ONLY ? A.compact_gate : nullptr);
}

template <typename D>
static cudaError_t launch_edges_and_points(const EaPrepArgs& A, cudaStream_t stream, int& nl) {
  const bool want_ref = (A.roles & EA_ROLE_REF) != 0;
  const bool gray = A.in_format != EA_IMAGE_BGR8;
  const size_t px0 = size_t(A.lv[0].w) * A.lv[0].h;
  const D* in_depth = static_cast<const D*>(A.in_depth);
  for (int l = 0; l < A.n_levels; ++l) {
    const EaPrepLevel& L = A.lv[l];
    const size_t pxl = size_t(L.w) * L.h;
    if (l > 0 && !edge_kernel_fuses_pyramid(A, l - 1)) {      // (otherwise level l - 1's edge kernel has already written this level)
      const EaPrepLevel& S = A.lv[l - 1];
      const EaImage sb = ea_level_image(A, l - 1);
      const D* sd = want_ref ? ((l == 1) ? in_depth : static_cast<const D*>(S.depth)) : nullptr;
      const size_t sstride = (l == 1) ? px0 : size_t(S.w) * S.h;
      const int32_t* sslots = (l == 1) ? nullptr : A.slots;
      D* dd = static_cast<D*>(L.depth);
      // one-channel input: planar rows that are 8-byte aligned (packed 4:2:2 takes the byte kernel)
      const bool vec4 = ((L.w & 3) == 0) && ((reinterpret_cast<uintptr_t>(sb.base) & 7) == 0) && ((reinterpret_cast<uintptr_t>(L.bgr) & 3) == 0) &&
                        (!gray || (sb.step == 1 && ((sb.stride | sb.pitch) & 7) == 0));
      if (vec4) {
        dim3 grid(unsigned((pxl / 4 + 255) / 256), unsigned(A.n));
        if (gray) k_pyr_down4<D, 1><<<grid, 256, 0, stream>>>(sb, sd, sstride, sslots, L.bgr, dd, A.slots, S.w, S.h);
        else k_pyr_down4<D, 3><<<grid, 256, 0, stream>>>(sb, sd, sstride, sslots, L.bgr, dd, A.slots, S.w, S.h);
      } else {
        dim3 grid(unsigned((pxl + 255) / 256), unsigned(A.n));
        if (gray) k_pyr_down<D, 1><<<grid, 256, 0, stream>>>(sb, sd, sstride, sslots, L.bgr, dd, A.slots, S.w, S.h);
        else k_pyr_down<D, 3><<<grid, 256, 0, stream>>>(sb, sd, sstride, sslots, L.bgr, dd, A.slots, S.w, S.h);
      }
      ++nl;
    }
    const EaImage b = ea_level_image(A, l);
    const D* d = want_ref ? ((l == 0) ? in_depth : static_cast<const D*>(L.depth)) : nullptr;
    const int32_t* ss = (l == 0) ? nullptr : A.slots;
    if (A.edge_detector != EA_EDGE_LAPLACIAN) {
      int k = 0;
      cudaError_t ce = ea_launch_canny_level(A, l, b, d, pxl, l != 0, A.canny, A.scratch, stream, &k);
      nl += k - 1;
      if (ce != cudaSuccess) return ce;
    } else if ((L.w & 3) == 0 && L.w >= 8 && L.h >= 4 && gray_words_ok(A, l)) {
      const bool fuse = edge_kernel_fuses_pyramid(A, l);
      uint8_t* nb = fuse ? A.lv[l + 1].bgr : nullptr;
      D* nd = (fuse && want_ref) ? static_cast<D*>(A.lv[l + 1].depth) : nullptr;
      if ((L.w % 128) != 0 && (L.w % 128) <= 64) {   // the last 128-wide tile would be at most half full: 64-wide tiles
        if (want_ref) launch_edge_mask2<D, 64, true>(A, L, b, d, pxl, ss, nb, nd, stream);
        else launch_edge_mask2<D, 64, false>(A, L, b, d, pxl, ss, nb, nd, stream);
      } else {
        if (want_ref) launch_edge_mask2<D, E2_TW, true>(A, L, b, d, pxl, ss, nb, nd, stream);
        else launch_edge_mask2<D, E2_TW, false>(A, L, b, d, pxl, ss, nb, nd, stream);
      }
    } else {   // generic byte path (any width)
      dim3 grid(unsigned((L.w + ET_W - 1) / ET_W), unsigned((L.h + ET_H - 1) / ET_H), unsigned(A.n));
      uint32_t* rb = want_ref ? L.ref_bits : nullptr;
      if (gray) k_edge_mask<D, 1><<<grid, dim3(ET_W, ET_H), 0, stream>>>(b, d, pxl, ss, A.slots, L.edge_bits, rb, L.w, L.h, L.words, A.grad_threshold, A.zero_to_one);
      else k_edge_mask<D, 3><<<grid, dim3(ET_W, ET_H), 0, stream>>>(b, d, pxl, ss, A.slots, L.edge_bits, rb, L.w, L.h, L.words, A.grad_threshold, A.zero_to_one);
    }
    ++nl;
    if (want_ref && A.in_mask) {
      k_mask_ref_bits<<<dim3(unsigned((L.h * L.words + 255) / 256), unsigned(A.n)), 256, 0, stream>>>(L.ref_bits, A.slots, A.in_mask, A.lv[0].w, A.lv[0].h, L.w, L.h, L.words, l, 0);
      ++nl;
    }
    if (A.in_now_mask) {
      k_mask_ref_bits<<<dim3(unsigned((L.h * L.words + 255) / 256), unsigned(A.n)), 256, 0, stream>>>(L.edge_bits, A.slots, A.in_now_mask, A.lv[0].w, A.lv[0].h, L.w, L.h, L.words, l, 1);
      ++nl;
    }
    if (want_ref && A.compact == EA_COMPACT_INLINE) {
      launch_compact<D>(A, l, stream);
      ++nl;
    }
  }
  return cudaGetLastError();
}

// edges, reference points and the median plane of A's frames
static cudaError_t launch_front(const EaPrepArgs& A, cudaStream_t stream, int& nl) {
  const bool want_now = (A.roles & EA_ROLE_NOW) != 0;
  cudaError_t pe = (A.depth_type == 1) ? launch_edges_and_points<float>(A, stream, nl) : launch_edges_and_points<uint16_t>(A, stream, nl);
  if (pe != cudaSuccess) return pe;
  if (want_now && A.dt_kind != EA_DT_EXACT && A.use_median) {
    const EaPrepLevel& L0 = A.lv[0];
    dim3 grid(unsigned((L0.h * L0.words + 255) / 256), unsigned(A.n), unsigned(A.n_levels));
    k_median_bits<<<grid, 256, 0, stream>>>(A);
    ++nl;
  }
  return cudaGetLastError();
}
// distance transforms of A's frames (now role)
static cudaError_t launch_dt(const EaPrepArgs& A, cudaStream_t stream, int& nl) {
  if (A.dt_kind == EA_DT_EXACT) {
    for (int l = 0; l < A.n_levels; ++l) {
      cudaError_t ee = ea_launch_exact_edt_level(A, l, A.scratch, stream, &nl);
      if (ee != cudaSuccess) return ee;
    }
    return cudaGetLastError();
  }
  const EaPrepLevel& L0 = A.lv[0];
  if (L0.w <= 32 * DTW_PMAX) {   // one warp per (frame, level); level 0 CTAs are scheduled first
    k_chamfer_dt_warp<<<dim3(unsigned(A.n), unsigned(A.n_levels)), 32, 0, stream>>>(A);
    ++nl;
    return cudaGetLastError();
  }
  // wider images: every level of every frame in one launch, CTA (frame, level); block sized for level 0
  const int P = (L0.w <= 4096) ? 4 : 8;
  const int threads = (((L0.w + P - 1) / P + 31) / 32) * 32;
  if (threads > 1024) return cudaErrorInvalidValue;
  dim3 grid(unsigned(A.n), unsigned(A.n_levels));
  if (P == 4) k_chamfer_dt<4><<<grid, threads, 0, stream>>>(A);
  else k_chamfer_dt<8><<<grid, threads, 0, stream>>>(A);
  ++nl;
  for (int l = 0; l < A.n_levels; ++l) { ea_launch_dt_fill_pad(A.lv[l], A.slots, A.n, stream); ++nl; }
  return cudaGetLastError();
}
// frames [f0, f0 + n) of A as an argument block of their own (pools are indexed by slot, inputs by frame)
static EaPrepArgs prep_slice(const EaPrepArgs& A, int f0, int n) {
  EaPrepArgs S = A;
  const size_t px0 = size_t(A.lv[0].w) * A.lv[0].h;
  S.n = n; S.slots = A.slots + f0;
  S.in_img = A.in_img + size_t(f0) * A.in_stride;
  if (A.in_depth) S.in_depth = static_cast<const char*>(A.in_depth) + size_t(f0) * px0 * (A.depth_type == 1 ? 4 : 2);
  if (A.in_mask) S.in_mask = A.in_mask + size_t(f0) * px0;
  if (A.in_now_mask) S.in_now_mask = A.in_now_mask + size_t(f0) * px0;
  return S;
}

static EaPrepArgs prep_args(const ea_frameset* fs, int n, const int32_t* d_slots, int roles, const EaFrameInput& in, int compact,
                            const ea_track_info* compact_gate) {
  const ea_frame_params& p = fs->p;
  EaPrepArgs A;
  std::memset(&A, 0, sizeof A);
  for (int l = 0; l < p.n_levels; ++l) A.lv[l] = fs->lv[l];
  A.n_levels = p.n_levels; A.slots = d_slots; A.in_img = in.image; A.in_depth = in.depth;
  // NV12 is its luma plane: the kernels read it as GRAY8 with the frame's pitch and stride
  A.in_format = in.layout.format == EA_IMAGE_NV12 ? EA_IMAGE_GRAY8 : in.layout.format;
  A.in_pitch = size_t(in.layout.row_pitch); A.in_stride = size_t(in.layout.frame_stride);
  A.in_mask = in.ref_mask; A.in_now_mask = in.now_mask;
  A.n_pts = fs->d_npts; A.dt_minmax = fs->d_minmax; A.dt_affine = fs->d_affine; A.overflow = fs->d_overflow;
  A.n = n; A.roles = roles; A.grad_threshold = p.grad_threshold; A.use_median = p.use_median;
  A.dt_normalize = p.dt_normalize;
  A.edge_detector = p.edge_detector; A.dt_kind = p.dt_kind;
  A.canny.low = p.canny_low; A.canny.high = p.canny_high; A.canny.l2 = p.canny_l2;
  A.canny.on_color = (p.edge_detector == EA_EDGE_CANNY_COLOR);
  A.scratch = fs->scratch;
  A.compact = compact; A.compact_gate = compact_gate;
  A.depth_type = p.depth_type; A.zero_to_one = p.zero_depth_to_one;
  A.depth_one = p.depth_type == EA_DEPTH_F32 ? 1.0f : float(p.depth_scale);
  if (A.edge_detector != EA_EDGE_LAPLACIAN) A.use_median = 0;   // the Canny pipelines of the reference have no median step
  return A;
}

// highest priority: the long-lived one-warp chamfer CTAs take the slots the short edge CTAs free, instead of queueing behind them
static int create_lanes(EaPrepPipe& P) {
  int pr_lo = 0, pr_hi = 0;
  CU(cudaDeviceGetStreamPriorityRange(&pr_lo, &pr_hi));
  for (int k = 0; k < EA_PREP_MAX_PARTS; ++k) {
    CU(cudaStreamCreateWithPriority(&P.aux[k], cudaStreamNonBlocking, pr_hi));
    CU(cudaEventCreateWithFlags(&P.ev_front[k], cudaEventDisableTiming));
    CU(cudaEventCreateWithFlags(&P.ev_dt[k], cudaEventDisableTiming));
  }
  P.ready = true;
  return EA_OK;
}

void ea_release_prep_lanes(ea_context* c) {
  EaPrepPipe& P = c->prep_pipe;
  for (int k = 0; k < EA_PREP_MAX_PARTS; ++k) {
    if (P.aux[k]) { cudaStreamSynchronize(P.aux[k]); cudaStreamDestroy(P.aux[k]); }
    if (P.ev_front[k]) cudaEventDestroy(P.ev_front[k]);
    if (P.ev_dt[k]) cudaEventDestroy(P.ev_dt[k]);
  }
  P = EaPrepPipe{};
}

// the whole pipeline for A's frames; lanes: null, or the auxiliary lanes that take the distance transforms of each half
static cudaError_t launch_pipeline(const EaPrepArgs& A, const EaPrepPipe* lanes, cudaStream_t stream, int& nl) {
  const bool want_ref = (A.roles & EA_ROLE_REF) != 0, want_now = (A.roles & EA_ROLE_NOW) != 0;
  if (want_ref && !A.in_depth) return cudaErrorInvalidValue;
  if (A.compact == EA_COMPACT_ONLY) {
    if (!want_ref || !A.compact_gate) return cudaErrorInvalidValue;
    for (int l = 0; l < A.n_levels; ++l) {
      if (A.depth_type == 1) launch_compact<float>(A, l, stream);
      else launch_compact<uint16_t>(A, l, stream);
      ++nl;
    }
    return cudaGetLastError();
  }
  cudaError_t e = cudaSuccess;
  if (!lanes) {
    e = launch_front(A, stream, nl);
    if (e == cudaSuccess && want_now) e = launch_dt(A, stream, nl);
  } else {
    const int K = EA_PREP_MAX_PARTS;
    int forked = 0;                                       // parts whose distance transforms are on their lane
    for (int k = 0; k < K && e == cudaSuccess; ++k) {
      const int f0 = int((long long)A.n * k / K), f1 = int((long long)A.n * (k + 1) / K);
      const EaPrepArgs H = prep_slice(A, f0, f1 - f0);
      e = launch_front(H, stream, nl);
      if (e != cudaSuccess) break;
      e = cudaEventRecord(lanes->ev_front[k], stream);
      if (e == cudaSuccess) e = cudaStreamWaitEvent(lanes->aux[k], lanes->ev_front[k], 0);
      if (e != cudaSuccess) break;
      forked = k + 1;
      e = launch_dt(H, lanes->aux[k], nl);
    }
    // join, also after an error: whatever reached a lane is ordered before the caller's next work on `stream`
    for (int k = 0; k < forked; ++k) {
      cudaError_t je = cudaEventRecord(lanes->ev_dt[k], lanes->aux[k]);
      if (je == cudaSuccess) je = cudaStreamWaitEvent(stream, lanes->ev_dt[k], 0);
      if (e == cudaSuccess) e = je;
    }
  }
  return e != cudaSuccess ? e : cudaGetLastError();
}

int ea_launch_preprocess(ea_frameset* fs, int n, const int32_t* d_slots, int roles, const EaFrameInput& in, cudaStream_t stream,
                         int compact, const ea_track_info* compact_gate) {
  ea_context* c = fs->ctx;
  const EaPrepArgs A = prep_args(fs, n, d_slots, roles, in, compact, compact_gate);
  // Two halves, two lanes: the chamfer kernel (DRAM- and latency-bound, ~40 % of the issue slots) of the first half runs beside
  // the edge kernels (issue-bound, a sixth of the DRAM bandwidth) of the second half.  Only the Laplacian + chamfer pipeline (its
  // work buffers are all indexed by slot), and only when both halves still fill the GPU: from 8 frames per SM (at 4 the halves
  // no longer fill it, DESIGN.md 4.4).
  const int split_frames_per_sm = 8;
  const bool split = compact != EA_COMPACT_ONLY && (roles & EA_ROLE_NOW) && A.edge_detector == EA_EDGE_LAPLACIAN &&
                     A.dt_kind != EA_DT_EXACT && A.lv[0].w <= 32 * DTW_PMAX && n >= split_frames_per_sm * c->sm_count;
  if (split && !c->prep_pipe.ready) {
    const int rc = create_lanes(c->prep_pipe);
    if (rc) return rc;
  }
  int nl = 0;
  EaProfileScope prof(c, 0, stream);
  const cudaError_t e = launch_pipeline(A, split ? &c->prep_pipe : nullptr, stream, nl);
  c->launches += nl;
  if (e != cudaSuccess) return ea_fail(EA_ERR_CUDA, "preprocess launch: %s", cudaGetErrorString(e));
  return EA_OK;
}

cudaError_t ea_launch_dt_normalized_copy(const float* origin, int pitch, const float2* affine, int w, int h, float* out, cudaStream_t stream) {
  k_dt_normalized_copy<<<(w * h + 255) / 256, 256, 0, stream>>>(origin, pitch, affine, w, h, out);
  return cudaGetLastError();
}
cudaError_t ea_launch_dt_import(const float* src, float* origin, int w, int h, int pitch, cudaStream_t stream) {
  const int n = pitch * (h + 2 * EA_DT_PAD);
  k_dt_import<<<(n + 255) / 256, 256, 0, stream>>>(src, origin, w, h, pitch);
  return cudaGetLastError();
}
cudaError_t ea_launch_dt_fill_pad(const EaPrepLevel& L, const int32_t* d_slots, int n, cudaStream_t stream) {
  const int tot = L.dt_pitch * (L.h + 2 * EA_DT_PAD);
  k_dt_fill_pad<<<dim3(unsigned(std::min((tot + 255) / 256, 1024)), unsigned(n)), 256, 0, stream>>>(L.dt, L.dt_slot, d_slots, L.w, L.h, L.dt_pitch);
  return cudaGetLastError();
}

cudaError_t ea_launch_unpack_mask(const uint32_t* bits, int w, int h, int words, int median, uint8_t* out, cudaStream_t stream) {
  k_unpack_mask<<<(w * h + 255) / 256, 256, 0, stream>>>(bits, w, h, words, median, out);
  return cudaGetLastError();
}
