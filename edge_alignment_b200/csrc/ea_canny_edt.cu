// Canny edge detector and exact Euclidean distance transform (the ROS-flavour preprocessing of the reference,
// src/SolveEA.cpp:46,102-109, and the standalone Canny variants standalone/utils.cpp:85-106, 371-462), batched.
// Bit-exact restatements of OpenCV's portable algorithms (canny.cpp, distransform.cpp trueDistTrans); pinned through
// the oracle against cv2 (tests/golden/cv2_stages.json).
#include "ea_internal.h"

namespace {

__device__ __forceinline__ int reflect101c(int i, int n) {
  if (n == 1) return 0;
  while (i < 0 || i >= n) i = (i < 0) ? -i : 2 * n - 2 - i;
  return i;
}
__device__ __forceinline__ int clampi(int i, int n) { return i < 0 ? 0 : (i >= n ? n - 1 : i); }

// cv::blur(3x3) (REFLECT_101, rounded /9) + cv::cvtColor(RGB2GRAY) on BGR data -> 8UC1   (utils.cpp:88-91)
// CN = 1: gray input, read where it lies (EaImage: the caller's luma at level 0); RGB2GRAY of three equal channels is the
// identity, so the blurred value is the output
template <int CN>
__global__ void __launch_bounds__(256) k_box_gray(const EaImage src, const int32_t* __restrict__ src_slots,
                                                  uint8_t* __restrict__ gray, size_t scratch_stride_px, int w, int h) {
  const int f = blockIdx.y;
  const uint8_t* img = src.base + (src_slots ? size_t(src_slots[f]) : size_t(f)) * src.stride + src.offset;
  uint8_t* out = gray + size_t(f) * scratch_stride_px;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < w * h; i += gridDim.x * blockDim.x) {
    const int x = i % w, y = i / w;
    int ch[CN];
#pragma unroll
    for (int c = 0; c < CN; ++c) {
      int acc = 0;
      for (int dy = -1; dy <= 1; ++dy) {
        const int yy = reflect101c(y + dy, h);
        for (int dx = -1; dx <= 1; ++dx) {
          if constexpr (CN == 3) acc += img[(size_t(yy) * w + reflect101c(x + dx, w)) * CN + c];
          else acc += img[size_t(yy) * src.pitch + size_t(reflect101c(x + dx, w)) * src.step];
        }
      }
      ch[c] = __double2int_rn(double(acc) * (1.0 / 9.0));
    }
    if constexpr (CN == 3) out[i] = uint8_t((ch[0] * 9798 + ch[1] * 19235 + ch[2] * 3735 + 16384) >> 15);
    else out[i] = uint8_t(ch[0]);
  }
}

// Sobel 3x3 (BORDER_REPLICATE) per channel, channel of largest magnitude (first on ties)   (canny.cpp)
// CN = 1: one channel read where it lies (EaImage: the caller's luma at level 0, or the blurred scratch plane)
template <int CN>
__global__ void __launch_bounds__(256) k_canny_grad(const EaImage src, const int32_t* __restrict__ src_slots,
                                                    bool slot_indexed, int* __restrict__ mag, short2* __restrict__ dxy,
                                                    size_t scratch_stride_px, int w, int h, int l2) {
  const int f = blockIdx.y;
  const uint8_t* img = src.base + ((slot_indexed && src_slots) ? size_t(src_slots[f]) : size_t(f)) * src.stride + src.offset;
  int* M = mag + size_t(f) * scratch_stride_px;
  short2* G = dxy + size_t(f) * scratch_stride_px;
  // byte of channel c of pixel (x, y)
  auto at = [&](int x, int y, int c) -> int {
    if constexpr (CN == 3) return img[(size_t(y) * w + x) * CN + c];
    else return img[size_t(y) * src.pitch + size_t(x) * src.step];
  };
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < w * h; i += gridDim.x * blockDim.x) {
    const int x = i % w, y = i / w;
    const int xm = clampi(x - 1, w), xp = clampi(x + 1, w), ym = clampi(y - 1, h), yp = clampi(y + 1, h);
    int best = -1, bdx = 0, bdy = 0;
#pragma unroll
    for (int c = 0; c < CN; ++c) {
      const int a = at(xm, ym, c), b = at(x, ym, c), cc = at(xp, ym, c);
      const int d = at(xm, y, c), e = at(xp, y, c);
      const int g = at(xm, yp, c), hh = at(x, yp, c), k = at(xp, yp, c);
      const int dx = (cc + 2 * e + k) - (a + 2 * d + g);
      const int dy = (g + 2 * hh + k) - (a + 2 * b + cc);
      const int m = l2 ? dx * dx + dy * dy : abs(dx) + abs(dy);
      if (m > best) { best = m; bdx = dx; bdy = dy; }
    }
    M[i] = best;
    G[i] = make_short2(short(bdx), short(bdy));
  }
}

// non-maximum suppression with the fixed-point tan(22.5 deg) test -> map: 1 = no edge, 0 = candidate, 2 = strong.  Each candidate or
// strong pixel also gets its union-find key for the hysteresis (hy_key) in lab, which is the dxy plane: the thread that reads pixel i's
// gradient is the one that overwrites it, after the read (the stored value depends on it).
__device__ __forceinline__ int hy_key(int i, bool strong, int n) { return strong ? i : n + i; }
__device__ __forceinline__ int hy_node(int key, int n) { return key >= n ? key - n : key; }

__global__ void __launch_bounds__(256) k_canny_nms(const int* __restrict__ mag, short2* dxy, uint8_t* __restrict__ map,
                                                   size_t scratch_stride_px, int w, int h, int low, int high) {
  const int f = blockIdx.y, n = w * h;
  const int* M = mag + size_t(f) * scratch_stride_px;
  short2* G = dxy + size_t(f) * scratch_stride_px;
  int* lab = reinterpret_cast<int*>(G);
  uint8_t* P = map + size_t(f) * scratch_stride_px;
  auto at = [&](int x, int y) { return (x < 0 || x >= w || y < 0 || y >= h) ? 0 : M[size_t(y) * w + x]; };
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const int x = i % w, y = i / w;
    const int m = M[i];
    bool is_max = false;
    if (m > low) {
      const int xs = G[i].x, ys = G[i].y;
      const int ax = abs(xs), ay = abs(ys) << 15;
      const int tg22x = ax * 13573;
      if (ay < tg22x) is_max = (m > at(x - 1, y) && m >= at(x + 1, y));
      else {
        const int tg67x = tg22x + (ax << 16);
        if (ay > tg67x) is_max = (m > at(x, y - 1) && m >= at(x, y + 1));
        else { const int sg = (xs ^ ys) < 0 ? -1 : 1; is_max = (m > at(x - sg, y - 1) && m > at(x + sg, y + 1)); }
      }
    }
    P[i] = is_max ? (m > high ? 2 : 0) : 1;
    if (is_max) lab[i] = hy_key(i, m > high, n);
  }
}

// ---- hysteresis: the edges are the candidate and strong pixels 8-connected to a strong one.  Union-find over those pixels: a node's
// entry in lab is the key of its parent, a root's is its own key.  Keys order strong pixels before candidates (hy_key), and a union
// always hangs the root with the larger key under the other, so a tree's root has its smallest key: the component holds a strong
// pixel iff its root key is < n.  Every entry only ever decreases (atomicMin) to the key of an ancestor, so concurrent unions and
// path halving keep every tree a tree of its component (the lock-free union of Playne & Hawick, 2018).  Work per pixel does not
// depend on how far along a chain the nearest strong pixel is.
__device__ __forceinline__ int hy_find(int* lab, int i, int n) {
  int k = __ldcg(lab + i);
  while (hy_node(k, n) != i) {
    const int p = hy_node(k, n), kp = __ldcg(lab + p);
    if (hy_node(kp, n) == p) return kp;
    atomicMin(lab + i, kp);                                     // path halving: i skips its parent
    i = hy_node(kp, n);
    k = __ldcg(lab + i);
  }
  return k;
}
__device__ __forceinline__ void hy_unite(int* lab, int a, int b, int n) {
  int ka = hy_find(lab, a, n), kb = hy_find(lab, b, n);
  while (ka != kb) {
    if (ka > kb) { const int t = ka; ka = kb; kb = t; }
    const int old = atomicMin(lab + hy_node(kb, n), ka);
    if (old == kb) return;                                      // kb was still a root: now under ka
    kb = hy_find(lab, hy_node(old, n), n);                      // kb was linked meanwhile: unite with its new root
  }
}

__global__ void __launch_bounds__(256) k_canny_union(const uint8_t* __restrict__ map, short2* dxy, size_t scratch_stride_px, int w, int h) {
  const int f = blockIdx.y, n = w * h;
  const uint8_t* P = map + size_t(f) * scratch_stride_px;
  int* lab = reinterpret_cast<int*>(dxy + size_t(f) * scratch_stride_px);
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    if (P[i] == 1) continue;
    const int x = i % w, y = i / w;
    // the neighbours before i in raster order (left, up-left, up, up-right); a pair of them that touch each other is united
    // by its own later pixel, so up alone, or left / up-left plus up-right, suffice
    const bool l = x > 0 && P[i - 1] != 1, ul = x > 0 && y > 0 && P[i - w - 1] != 1, u = y > 0 && P[i - w] != 1,
               ur = x + 1 < w && y > 0 && P[i - w + 1] != 1;
    if (u) { hy_unite(lab, i, i - w, n); continue; }
    if (l) hy_unite(lab, i, i - 1, n);
    else if (ul) hy_unite(lab, i, i - w - 1, n);
    if (ur) hy_unite(lab, i, i - w + 1, n);
  }
}

// edge = candidate or strong pixel whose root key is a strong pixel's; packs the edge plane and the reference plane (edge with depth,
// or every edge with zero_to_one), one warp per 32-pixel word
template <typename D>
__global__ void __launch_bounds__(256) k_canny_pack(const uint8_t* __restrict__ map, const short2* dxy, size_t scratch_stride_px,
                                                    const D* __restrict__ depth, size_t depth_stride_px, const int32_t* __restrict__ depth_slots,
                                                    bool depth_slot_indexed, const int32_t* __restrict__ dst_slots, uint32_t* __restrict__ edge_bits,
                                                    uint32_t* __restrict__ ref_bits, int w, int h, int words, int zero_to_one) {
  const int f = blockIdx.y, n = w * h;
  const uint8_t* P = map + size_t(f) * scratch_stride_px;
  const int* lab = reinterpret_cast<const int*>(dxy + size_t(f) * scratch_stride_px);
  const D* dep = depth ? depth + ((depth_slot_indexed && depth_slots) ? size_t(depth_slots[f]) : size_t(f)) * depth_stride_px : nullptr;
  const size_t obase = size_t(dst_slots[f]) * h * words;
  const int total = h * words * 32;                           // a multiple of 32: every warp's pixels fall in one word
  for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < total; t += gridDim.x * blockDim.x) {
    const int y = t / (words * 32), x = t % (words * 32);
    bool edge = false, ref = false;
    if (x < w) {
      const int i = y * w + x;
      if (P[i] != 1) {
        int j = i, k = lab[i];
        while (hy_node(k, n) != j) { j = hy_node(k, n); k = lab[j]; }
        edge = k < n;
        ref = edge && dep && (zero_to_one || dep[i] > D(0));
      }
    }
    const unsigned eb = __ballot_sync(0xffffffffu, edge), rb = __ballot_sync(0xffffffffu, ref);
    if ((threadIdx.x & 31) == 0) {
      edge_bits[obase + (t >> 5)] = eb;
      if (ref_bits) ref_bits[obase + (t >> 5)] = rb;
    }
  }
}

// ---- exact Euclidean DT (trueDistTrans): column pass -> vertical distance (1<<20 == none), row pass -> exact integer
// minimum of (q-p)^2 + g(p)^2 searched outwards until k^2 can no longer win, then sqrtf -----------------------------------
#define EDT_INF (1 << 20)
__global__ void __launch_bounds__(256) k_edt_cols(const uint32_t* __restrict__ edge_bits, const int32_t* __restrict__ dst_slots,
                                                  int* __restrict__ g, size_t scratch_stride_px, int w, int h, int words) {
  const int f = blockIdx.y;
  const uint32_t* bits = edge_bits + size_t(dst_slots[f]) * h * words;
  int* G = g + size_t(f) * scratch_stride_px;
  const int x = blockIdx.x * blockDim.x + threadIdx.x;
  if (x >= w) return;
  int dist = EDT_INF;
  for (int y = h - 1; y >= 0; --y) {
    const bool z = (bits[size_t(y) * words + (x >> 5)] >> (x & 31)) & 1u;     // edge pixel == zero pixel of the inverted map
    dist = z ? 0 : min(dist + 1, EDT_INF);
    G[size_t(y) * w + x] = dist;
  }
  dist = EDT_INF;
  for (int y = 0; y < h; ++y) {
    const bool z = (bits[size_t(y) * words + (x >> 5)] >> (x & 31)) & 1u;
    dist = z ? 0 : min(dist + 1, EDT_INF);
    G[size_t(y) * w + x] = min(G[size_t(y) * w + x], dist);
  }
}

__global__ void __launch_bounds__(256) k_edt_rows(const int* __restrict__ g, size_t scratch_stride_px, const int32_t* __restrict__ dst_slots,
                                                  float* __restrict__ dt, size_t dt_slot, int pitch, unsigned* __restrict__ fminmax, int level, int w, int h) {
  const int f = blockIdx.y, slot = dst_slots[f];
  const int* G = g + size_t(f) * scratch_stride_px;
  float* D = dt + size_t(slot) * dt_slot + size_t(EA_DT_PAD) * pitch + EA_DT_PAD;   // pixel (0,0) of the padded image
  unsigned lmin = 0x7F800000u, lmax = 0u;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < w * h; i += gridDim.x * blockDim.x) {
    const int q = i % w;
    const int* row = G + size_t(i / w) * w;
    long long best = -1;
    const int g0 = row[q];
    if (g0 < EDT_INF) best = (long long)g0 * g0;
    for (int k = 1; k < w; ++k) {
      const long long kk = (long long)k * k;
      if (best >= 0 && kk >= best) break;
      if (q - k < 0 && q + k >= w) break;
      if (q - k >= 0) { const int a = row[q - k]; if (a < EDT_INF) { const long long v = kk + (long long)a * a; if (best < 0 || v < best) best = v; } }
      if (q + k < w) { const int a = row[q + k]; if (a < EDT_INF) { const long long v = kk + (long long)a * a; if (best < 0 || v < best) best = v; } }
    }
    const float r = best < 0 ? 65536.0f : __fsqrt_rn(float(best));
    D[size_t(i / w) * pitch + q] = r;
    const unsigned bits = __float_as_uint(r);
    lmin = min(lmin, bits); lmax = max(lmax, bits);
  }
  lmin = __reduce_min_sync(0xffffffffu, lmin); lmax = __reduce_max_sync(0xffffffffu, lmax);
  if ((threadIdx.x & 31) == 0) { atomicMin(&fminmax[(slot * EA_MAX_LEVELS + level) * 2], lmin); atomicMax(&fminmax[(slot * EA_MAX_LEVELS + level) * 2 + 1], lmax); }
}

__global__ void k_edt_minmax_init(unsigned* fminmax, const int32_t* dst_slots, int level, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) { fminmax[(dst_slots[i] * EA_MAX_LEVELS + level) * 2] = 0x7F800000u; fminmax[(dst_slots[i] * EA_MAX_LEVELS + level) * 2 + 1] = 0u; }
}
__global__ void k_edt_affine(const unsigned* fminmax, const int32_t* dst_slots, int level, int n, int dt_normalize, float2* affine) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int slot = dst_slots[i];
  float2 aff = make_float2(1.0f, 0.0f);
  if (dt_normalize != EA_NORM_NONE) {
    const double beta = (dt_normalize == EA_NORM_255) ? 255.0 : 1.0;
    const float fmn = __uint_as_float(fminmax[(slot * EA_MAX_LEVELS + level) * 2]), fmx = __uint_as_float(fminmax[(slot * EA_MAX_LEVELS + level) * 2 + 1]);
    const double range = double(fmx) - double(fmn);
    const double scale = beta * (range > 2.220446049250313e-16 ? 1.0 / range : 0.0);
    aff = make_float2(float(scale), float(0.0 - double(fmn) * scale));
  }
  affine[slot * EA_MAX_LEVELS + level] = aff;
}

}  // namespace

// Edge planes of level l by Canny.  img = BGR (or one-channel input's luma) of that level; depth is dense, frame_stride_px pixels
// per frame.  scratch: gray u8 | mag i32 | dxy short2 | map u8, each [n][stride] with stride = level-0 pixels.
cudaError_t ea_launch_canny_level(const EaPrepArgs& A, int l, const EaImage& img, const void* depth, size_t frame_stride_px,
                                  bool slot_indexed, const EaCannyCfg& cfg, const EaScratch& S, cudaStream_t stream, int* launches) {
  const EaPrepLevel& L = A.lv[l];
  const int npx = L.w * L.h;
  if (npx > (1 << 30)) return cudaErrorInvalidValue;              // the hysteresis' union-find keys go up to 2 w h
  dim3 grid(unsigned(std::min((npx + 255) / 256, 4096)), unsigned(A.n));
  double t1 = cfg.low, t2 = cfg.high;
  if (t1 > t2) { const double t = t1; t1 = t2; t2 = t; }
  if (cfg.l2) {
    t1 = std::min(32767.0, t1); t2 = std::min(32767.0, t2);
    if (t1 > 0) t1 *= t1;
    if (t2 > 0) t2 *= t2;
  }
  const int low = int(floor(t1)), high = int(floor(t2));
  if (cfg.on_color) {
    // on gray input the channel of largest gradient (first on ties) of (g, g, g) is g itself
    if (A.in_format != EA_IMAGE_BGR8) k_canny_grad<1><<<grid, 256, 0, stream>>>(img, A.slots, slot_indexed, S.mag, S.dxy, S.stride, L.w, L.h, cfg.l2);
    else k_canny_grad<3><<<grid, 256, 0, stream>>>(img, A.slots, slot_indexed, S.mag, S.dxy, S.stride, L.w, L.h, cfg.l2);
    ++*launches;
  } else {
    if (A.in_format != EA_IMAGE_BGR8) k_box_gray<1><<<grid, 256, 0, stream>>>(img, slot_indexed ? A.slots : nullptr, S.gray, S.stride, L.w, L.h);
    else k_box_gray<3><<<grid, 256, 0, stream>>>(img, slot_indexed ? A.slots : nullptr, S.gray, S.stride, L.w, L.h);
    const EaImage blurred{S.gray, S.stride, size_t(L.w), 1, 0};
    k_canny_grad<1><<<grid, 256, 0, stream>>>(blurred, nullptr, false, S.mag, S.dxy, S.stride, L.w, L.h, cfg.l2);
    *launches += 2;
  }
  k_canny_nms<<<grid, 256, 0, stream>>>(S.mag, S.dxy, S.map, S.stride, L.w, L.h, low, high);
  k_canny_union<<<grid, 256, 0, stream>>>(S.map, S.dxy, S.stride, L.w, L.h);
  const int npack = L.h * L.words * 32;
  const dim3 pgrid(unsigned(std::min((npack + 255) / 256, 4096)), unsigned(A.n));
  const bool want_ref = (A.roles & EA_ROLE_REF) != 0;
  if (A.depth_type == 1)
    k_canny_pack<float><<<pgrid, 256, 0, stream>>>(S.map, S.dxy, S.stride, want_ref ? static_cast<const float*>(depth) : nullptr, frame_stride_px, A.slots,
                                                   slot_indexed, A.slots, L.edge_bits, want_ref ? L.ref_bits : nullptr, L.w, L.h, L.words, A.zero_to_one);
  else
    k_canny_pack<uint16_t><<<pgrid, 256, 0, stream>>>(S.map, S.dxy, S.stride, want_ref ? static_cast<const uint16_t*>(depth) : nullptr, frame_stride_px,
                                                      A.slots, slot_indexed, A.slots, L.edge_bits, want_ref ? L.ref_bits : nullptr, L.w, L.h, L.words,
                                                      A.zero_to_one);
  *launches += 3;
  return cudaGetLastError();
}

cudaError_t ea_launch_exact_edt_level(const EaPrepArgs& A, int l, const EaScratch& S, cudaStream_t stream, int* launches) {
  const EaPrepLevel& L = A.lv[l];
  const int npx = L.w * L.h;
  k_edt_minmax_init<<<(A.n + 255) / 256, 256, 0, stream>>>(A.dt_minmax, A.slots, l, A.n);
  k_edt_cols<<<dim3(unsigned((L.w + 255) / 256), unsigned(A.n)), 256, 0, stream>>>(L.edge_bits, A.slots, S.mag, S.stride, L.w, L.h, L.words);
  k_edt_rows<<<dim3(unsigned(std::min((npx + 255) / 256, 4096)), unsigned(A.n)), 256, 0, stream>>>(S.mag, S.stride, A.slots, L.dt, L.dt_slot, L.dt_pitch, A.dt_minmax, l, L.w, L.h);
  k_edt_affine<<<(A.n + 255) / 256, 256, 0, stream>>>(A.dt_minmax, A.slots, l, A.n, A.dt_normalize, A.dt_affine);
  ea_launch_dt_fill_pad(L, A.slots, A.n, stream);
  *launches += 5;
  return cudaGetLastError();
}
