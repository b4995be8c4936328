// Front-end kernels of the B200 AprilTag engine (sm_100a):
//   K1  gray conversion + decimation + 4x4 tile min/max      (reference: threshold.cu:16-80)
//   K1b Gaussian quad_sigma filter                            (upstream image_u8_gaussian_blur)
//   K2  3x3 tile min/max dilation + adaptive threshold        (threshold.cu:84-147)
//   K3  tile-local union-find in shared memory                (labeling_allegretti_2019_BKE.cu:114-300)
//   K4  cross-tile merge with global atomicMin                (:302-338)
//   K5  pointer-jumping compression + component sizes         (:287-300,340-462)
//   K6  boundary points, ballot/match compaction, blob-pair hash with extents
//                                                            (apriltag_gpu.cu:226-360,788-862)
// All integer work: bit-exact against oracle/ by construction.  No tensor cores: nothing
// here is a contraction; the bound is HBM/L2 bandwidth and atomics latency.
#include <cuda_runtime.h>
#include <stdint.h>

#include "dev_types.h"
#include "kernels.h"

namespace b200tag {

// ---------------------------------------------------------------------------------------------
// K1: YUYV, decimate 2.  One thread = one threshold tile = 8x8 full-res pixels (128 B of YUYV):
// eight independent 16-byte loads in flight per thread, 8-byte gray stores, 4-byte quad stores.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) k_pre_yuyv_dec2(FrameParams p) {
  const int tx = blockIdx.x * blockDim.x + threadIdx.x;
  const int ty = blockIdx.y;
  const int frame = blockIdx.z;
  if (tx >= p.tiles_x) return;
  const size_t N = static_cast<size_t>(p.W) * p.H, n = static_cast<size_t>(p.w) * p.h;
  const uint8_t *in = p.in + frame * p.in_stride;
  uint8_t *gray = p.gray + frame * N;
  uint8_t *quad = p.quad + frame * n;
  uint4 v[8];
#pragma unroll
  for (int r = 0; r < 8; r++) {
    const size_t row = static_cast<size_t>(ty) * 8 + r;
    v[r] = __ldcs(reinterpret_cast<const uint4 *>(in + (row * p.W + static_cast<size_t>(tx) * 8) * 2));
  }
  uint32_t mn = 0xffffffffu, mx = 0;
#pragma unroll
  for (int r = 0; r < 8; r++) {
    const size_t row = static_cast<size_t>(ty) * 8 + r;
    const uint32_t lo = __byte_perm(v[r].x, v[r].y, 0x6420);
    const uint32_t hi = __byte_perm(v[r].z, v[r].w, 0x6420);
    *reinterpret_cast<uint2 *>(gray + row * p.W + static_cast<size_t>(tx) * 8) = make_uint2(lo, hi);
    if ((r & 1) == 0) {
      const uint32_t d = __byte_perm(lo, hi, 0x6420);
      const size_t qrow = static_cast<size_t>(ty) * 4 + (r >> 1);
      *reinterpret_cast<uint32_t *>(quad + qrow * p.w + static_cast<size_t>(tx) * 4) = d;
      mn = __vminu4(mn, d);
      mx = __vmaxu4(mx, d);
    }
  }
  mn = __vminu4(mn, mn >> 16);
  mn = __vminu4(mn, mn >> 8);
  mx = __vmaxu4(mx, mx >> 16);
  mx = __vmaxu4(mx, mx >> 8);
  uint8_t *mm = p.minmax_raw + (frame * static_cast<size_t>(p.tiles_x) * p.tiles_y + static_cast<size_t>(ty) * p.tiles_x + tx) * 2;
  *reinterpret_cast<uchar2 *>(mm) = make_uchar2(mn & 0xff, mx & 0xff);
}

// K1 for GRAY8 input, decimate 2 (the gray image is the caller's buffer, nothing to write back):
// one thread = one threshold tile; only the even rows are read, 8 bytes each.
__global__ void __launch_bounds__(128) k_pre_gray_dec2(FrameParams p) {
  const int tx = blockIdx.x * blockDim.x + threadIdx.x;
  const int ty = blockIdx.y;
  const int frame = blockIdx.z;
  if (tx >= p.tiles_x) return;
  const size_t n = static_cast<size_t>(p.w) * p.h;
  const uint8_t *in = p.in + frame * p.in_stride;
  uint8_t *quad = p.quad + frame * n;
  uint2 v[4];
#pragma unroll
  for (int r = 0; r < 4; r++) {
    const size_t row = static_cast<size_t>(ty) * 8 + 2 * r;
    v[r] = __ldcs(reinterpret_cast<const uint2 *>(in + row * p.W + static_cast<size_t>(tx) * 8));
  }
  uint32_t mn = 0xffffffffu, mx = 0;
#pragma unroll
  for (int r = 0; r < 4; r++) {
    const uint32_t d = __byte_perm(v[r].x, v[r].y, 0x6420);
    *reinterpret_cast<uint32_t *>(quad + (static_cast<size_t>(ty) * 4 + r) * p.w + static_cast<size_t>(tx) * 4) = d;
    mn = __vminu4(mn, d);
    mx = __vmaxu4(mx, d);
  }
  mn = __vminu4(mn, mn >> 16);
  mn = __vminu4(mn, mn >> 8);
  mx = __vmaxu4(mx, mx >> 16);
  mx = __vmaxu4(mx, mx >> 8);
  uint8_t *mm = p.minmax_raw + (frame * static_cast<size_t>(p.tiles_x) * p.tiles_y + static_cast<size_t>(ty) * p.tiles_x + tx) * 2;
  *reinterpret_cast<uchar2 *>(mm) = make_uchar2(mn & 0xff, mx & 0xff);
}

__device__ __forceinline__ uint8_t luma_of(const uint8_t *in, int fmt, size_t i) {
  if (fmt == B200TAG_FMT_GRAY8) return in[i];
  if (fmt == B200TAG_FMT_YUYV) return in[2 * i];
  const int b = in[3 * i], g = in[3 * i + 1], r = in[3 * i + 2];
  // Y of cv::COLOR_BGR2YUV_YUYV, the conversion the node applies before Detect
  // (apriltags_cuda_detector.cu:401)
  return static_cast<uint8_t>((4211 * r + 8258 * g + 1606 * b + (1 << 13) + (16 << 14)) >> 14);
}

// K1 for BGR8 input, decimate 2 -- the node's own frames (sensor_msgs bgr8, quad_decimate 2,
// apriltags_cuda_detector.cu:399-404) without the CPU cvtColor: one thread = one threshold tile = 8x8 input
// pixels = 24 bytes per row, read as three 8-byte words; luma as cv::COLOR_BGR2YUV_YUYV computes it.
__global__ void __launch_bounds__(128) k_pre_bgr_dec2(FrameParams p) {
  const int tx = blockIdx.x * blockDim.x + threadIdx.x;
  const int ty = blockIdx.y;
  const int frame = blockIdx.z;
  if (tx >= p.tiles_x) return;
  const size_t N = static_cast<size_t>(p.W) * p.H, n = static_cast<size_t>(p.w) * p.h;
  const uint8_t *in = p.in + frame * p.in_stride;
  uint8_t *gray = p.gray + frame * N;
  uint8_t *quad = p.quad + frame * n;
  uint32_t mn = 0xffffffffu, mx = 0;
#pragma unroll
  for (int half = 0; half < 2; half++) {
    uint2 v[4][3];
#pragma unroll
    for (int r = 0; r < 4; r++) {
      const size_t row = static_cast<size_t>(ty) * 8 + half * 4 + r;
      const uint2 *src = reinterpret_cast<const uint2 *>(in + (row * p.W + static_cast<size_t>(tx) * 8) * 3);
      v[r][0] = __ldcs(src);
      v[r][1] = __ldcs(src + 1);
      v[r][2] = __ldcs(src + 2);
    }
#pragma unroll
    for (int r = 0; r < 4; r++) {
      const size_t row = static_cast<size_t>(ty) * 8 + half * 4 + r;
      const uint32_t wds[6] = {v[r][0].x, v[r][0].y, v[r][1].x, v[r][1].y, v[r][2].x, v[r][2].y};
      uint32_t out[2] = {0, 0};
#pragma unroll
      for (int px = 0; px < 8; px++) {
        const int byte = px * 3;
        const uint32_t bb = (wds[byte >> 2] >> ((byte & 3) * 8)) & 0xff;
        const uint32_t gg = (wds[(byte + 1) >> 2] >> (((byte + 1) & 3) * 8)) & 0xff;
        const uint32_t rr = (wds[(byte + 2) >> 2] >> (((byte + 2) & 3) * 8)) & 0xff;
        const uint32_t y = (4211u * rr + 8258u * gg + 1606u * bb + (1u << 13) + (16u << 14)) >> 14;
        out[px >> 2] |= y << (8 * (px & 3));
      }
      *reinterpret_cast<uint2 *>(gray + row * p.W + static_cast<size_t>(tx) * 8) = make_uint2(out[0], out[1]);
      if ((r & 1) == 0) {
        const uint32_t d = __byte_perm(out[0], out[1], 0x6420);
        const size_t qrow = static_cast<size_t>(ty) * 4 + half * 2 + (r >> 1);
        *reinterpret_cast<uint32_t *>(quad + qrow * p.w + static_cast<size_t>(tx) * 4) = d;
        mn = __vminu4(mn, d);
        mx = __vmaxu4(mx, d);
      }
    }
  }
  mn = __vminu4(mn, mn >> 16);
  mn = __vminu4(mn, mn >> 8);
  mx = __vmaxu4(mx, mx >> 16);
  mx = __vmaxu4(mx, mx >> 8);
  uint8_t *mm = p.minmax_raw + (frame * static_cast<size_t>(p.tiles_x) * p.tiles_y + static_cast<size_t>(ty) * p.tiles_x + tx) * 2;
  *reinterpret_cast<uchar2 *>(mm) = make_uchar2(mn & 0xff, mx & 0xff);
}

// K1 generic: any format, any integer decimation.  One thread = one threshold tile
// (4f x 4f full-res pixels).  `dst_quad` is quad_tmp when a blur follows.
__global__ void __launch_bounds__(128) k_pre_generic(FrameParams p, int write_minmax) {
  const int tx = blockIdx.x * blockDim.x + threadIdx.x;
  const int ty = blockIdx.y;
  const int frame = blockIdx.z;
  if (tx >= p.tiles_x) return;
  const size_t N = static_cast<size_t>(p.W) * p.H, n = static_cast<size_t>(p.w) * p.h;
  const uint8_t *in = p.in + frame * p.in_stride;
  uint8_t *gray = p.gray + frame * N;
  uint8_t *quad = (p.blur_ksz ? p.quad_tmp : p.quad) + frame * n;
  const int f = p.f, span = 4 * f;
  int mn = 255, mx = 0;
  for (int r = 0; r < span; r++) {
    const size_t row = static_cast<size_t>(ty) * span + r;
    for (int c = 0; c < span; c++) {
      const size_t col = static_cast<size_t>(tx) * span + c;
      const uint8_t g = luma_of(in, p.fmt, row * p.W + col);
      if (p.fmt != B200TAG_FMT_GRAY8) gray[row * p.W + col] = g;
      if ((r % f) == 0 && (c % f) == 0) {
        quad[(row / f) * p.w + col / f] = g;
        mn = min(mn, static_cast<int>(g));
        mx = max(mx, static_cast<int>(g));
      }
    }
  }
  if (write_minmax) {
    uint8_t *mm = p.minmax_raw + (frame * static_cast<size_t>(p.tiles_x) * p.tiles_y + static_cast<size_t>(ty) * p.tiles_x + tx) * 2;
    mm[0] = static_cast<uint8_t>(mn);
    mm[1] = static_cast<uint8_t>(mx);
  }
}

// K1 for GRAY8 / BGR8 at decimate 1 with 16-byte accesses: one thread = 16 pixels of one row.
// (config 3's input shape; tile min/max is computed by k_tile_minmax afterwards.)
__global__ void __launch_bounds__(256) k_pre_bgr_dec1(FrameParams p) {
  const size_t N = static_cast<size_t>(p.W) * p.H;
  const int frame = blockIdx.y;
  const size_t g16 = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;  // group of 16 pixels
  if (g16 * 16 >= N) return;
  const uint8_t *in = p.in + frame * p.in_stride;
  const uint4 *src = reinterpret_cast<const uint4 *>(in + g16 * 48);
  const uint4 a = __ldcs(src), b = __ldcs(src + 1), c = __ldcs(src + 2);
  const uint32_t wds[12] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w, c.x, c.y, c.z, c.w};
  uint32_t out[4];
#pragma unroll
  for (int q = 0; q < 4; q++) {
    uint32_t o = 0;
#pragma unroll
    for (int k = 0; k < 4; k++) {
      const int px = q * 4 + k, byte = px * 3;
      const uint32_t bb = (wds[byte >> 2] >> ((byte & 3) * 8)) & 0xff;
      const uint32_t gg = (wds[(byte + 1) >> 2] >> (((byte + 1) & 3) * 8)) & 0xff;
      const uint32_t rr = (wds[(byte + 2) >> 2] >> (((byte + 2) & 3) * 8)) & 0xff;
      const uint32_t y = (4211u * rr + 8258u * gg + 1606u * bb + (1u << 13) + (16u << 14)) >> 14;
      o |= y << (8 * k);
    }
    out[q] = o;
  }
  const uint4 o4 = make_uint4(out[0], out[1], out[2], out[3]);
  *reinterpret_cast<uint4 *>(p.gray + frame * N + g16 * 16) = o4;
  uint8_t *quad = (p.blur_ksz ? p.quad_tmp : p.quad) + frame * N;
  *reinterpret_cast<uint4 *>(quad + g16 * 16) = o4;
}

// K1b: separable Gaussian with upstream's border rule (convolve(): indices [ksz/2, sz-ksz+ksz/2) are filtered, the
// rest copied), rows first then columns.  One CTA = 64x128 output pixels (64x32: 0.066 ms per 16 config-3 frames, 64x128: 0.061).  The input tile with its halo is staged in
// shared memory with 4-byte loads (the halo is rounded up to a multiple of 4 columns so every word is aligned); both
// passes work on words: a thread filters 4 neighbouring pixels from the bytes it has in registers (row pass) or from
// aligned word loads of the rows above and below (column pass) and stores one word.  Runs the filter lengths that
// k_blur_strip does not take.
constexpr int kBlurTW = 64, kBlurTH = 128;  // (the host caps the filter radius at 15: detector.cu blur_kernel)
__global__ void __launch_bounds__(256) k_blur(FrameParams p) {
  extern __shared__ __align__(16) uint8_t s_blur[];
  const int ksz = p.blur_ksz, r = ksz >> 1, r4 = (r + 3) & ~3;
  const int sw = kBlurTW + 2 * r4, sh = kBlurTH + 2 * r;   // staged input tile, sw a multiple of 4
  uint8_t *s_in = s_blur;                                   // [sh][sw]
  uint8_t *s_row = s_blur + sh * sw;                        // [sh][kBlurTW]: row-filtered
  const int x0 = blockIdx.x * kBlurTW, y0 = blockIdx.y * kBlurTH;
  const int frame = blockIdx.z;
  const size_t n = static_cast<size_t>(p.w) * p.h;
  const uint8_t *src = p.quad_tmp + frame * n;
  uint8_t *dst = p.quad + frame * n;
  const int lane = threadIdx.x & 31, wrp = threadIdx.x >> 5;
  // stage: warp = row (stride 8), lane = word of the row
  for (int yy = wrp; yy < sh; yy += 8) {
    const int gy = y0 - r + yy;
    for (int cw = lane; cw < sw / 4; cw += 32) {
      const int gx = x0 - r4 + 4 * cw;
      uint32_t v = 0;
      if (gy >= 0 && gy < p.h && gx >= 0 && gx < p.w) v = __ldg(reinterpret_cast<const uint32_t *>(src + static_cast<size_t>(gy) * p.w + gx));
      reinterpret_cast<uint32_t *>(s_in + yy * sw)[cw] = v;
    }
  }
  __syncthreads();
  // row pass: thread = 4 pixels of a staged row (16 words per row, 16 rows per sweep)
  const int q = threadIdx.x & 15, rsub = threadIdx.x >> 4;
  for (int yy = rsub; yy < sh; yy += 16) {
    const uint8_t *row = s_in + yy * sw + r4 + 4 * q;   // the thread's first pixel
    uint32_t out = 0;
#pragma unroll
    for (int px = 0; px < 4; px++) {
      const int gx = x0 + 4 * q + px;
      uint32_t v = row[px];
      if (gx >= r && gx < p.w - ksz + r) {
        uint32_t acc = 0;
        for (int j = 0; j < ksz; j++) acc += static_cast<uint32_t>(p.blur_k[j]) * row[px - r + j];
        v = (acc >> 8) & 0xff;
      }
      out |= v << (8 * px);
    }
    reinterpret_cast<uint32_t *>(s_row + yy * kBlurTW)[q] = out;
  }
  __syncthreads();
  // column pass: thread = one word of an output row, aligned word loads of the ksz rows it needs
  for (int yy = rsub; yy < kBlurTH; yy += 16) {
    const int gx = x0 + 4 * q, gy = y0 + yy;
    if (gx >= p.w || gy >= p.h) continue;
    uint32_t out = reinterpret_cast<const uint32_t *>(s_row + (yy + r) * kBlurTW)[q];
    if (gy >= r && gy < p.h - ksz + r) {
      uint32_t a0 = 0, a1 = 0, a2 = 0, a3 = 0;
      for (int j = 0; j < ksz; j++) {
        const uint32_t wv = reinterpret_cast<const uint32_t *>(s_row + (yy + j) * kBlurTW)[q], kj = p.blur_k[j];
        a0 += kj * (wv & 0xff); a1 += kj * ((wv >> 8) & 0xff); a2 += kj * ((wv >> 16) & 0xff); a3 += kj * (wv >> 24);
      }
      out = ((a0 >> 8) & 0xff) | (((a1 >> 8) & 0xff) << 8) | (((a2 >> 8) & 0xff) << 16) | (((a3 >> 8) & 0xff) << 24);
    }
    if (p.sharpen) {
      const uint32_t orig = reinterpret_cast<const uint32_t *>(s_in + (yy + r) * sw + r4)[q];
      uint32_t o = 0;
#pragma unroll
      for (int px = 0; px < 4; px++) {
        int sv = 2 * static_cast<int>((orig >> (8 * px)) & 0xff) - static_cast<int>((out >> (8 * px)) & 0xff);
        sv = max(0, min(255, sv));
        o |= static_cast<uint32_t>(sv) << (8 * px);
      }
      out = o;
    }
    *reinterpret_cast<uint32_t *>(dst + static_cast<size_t>(gy) * p.w + gx) = out;
  }
}

// K1b for filter lengths 3, 5, 7 (quad_sigma up to 1.9) without shared memory: a warp owns a strip of 32 words (128
// pixels) x kBlurRows rows and walks down it.  Per input row a lane loads ONE aligned word, takes its neighbours' words by
// shuffle (the strip's edge lanes load theirs), forms the byte-shifted words of the taps with funnel shifts and filters
// the even and the odd bytes as two 16-bit lanes of a 32-bit multiply-add (the taps sum to at most 255, so a lane never
// exceeds 255 * 255); the row-filtered words of the last KSZ rows stay in registers, unpacked, and the column pass of
// the row in their middle is KSZ more multiply-adds.  Same border rule and arithmetic as k_blur.
constexpr int kBlurRows = 32, kBlurAhead = 4;  // (64 rows with 8 rows ahead: 0.055 ms against 0.049 per 16 config-3 frames)
static_assert(kBlurRows % 4 == 0, "strips start on tile rows");
template <int KSZ>
__global__ void __launch_bounds__(128) k_blur_strip(FrameParams p) {
  constexpr int R = KSZ / 2;
  static_assert(KSZ == 3 || KSZ == 5 || KSZ == 7, "one neighbour word on each side covers the taps");
  const int lane = threadIdx.x & 31, wrp = threadIdx.x >> 5;
  const int frame = blockIdx.z;
  const int ww = p.w >> 2;  // words per row
  const int wx = blockIdx.x * 32 + lane;
  const int gy0 = (blockIdx.y * 4 + wrp) * kBlurRows;
  if (gy0 >= p.h) return;  // (warp-uniform)
  const size_t n = static_cast<size_t>(p.w) * p.h;
  const uint32_t *src = reinterpret_cast<const uint32_t *>(p.quad_tmp + frame * n);
  uint32_t *dst = reinterpret_cast<uint32_t *>(p.quad + frame * n);
  const bool in_x = wx < ww;
  const int ex = lane == 0 ? wx - 1 : wx + 1;  // the word an edge lane fetches for its missing neighbour
  const bool has_ex = (lane == 0 || lane == 31) && ex >= 0 && ex < ww;
  uint32_t xmask = 0;  // bytes that the row pass filters (the others are copied)
#pragma unroll
  for (int k = 0; k < 4; k++) {
    const int gx = 4 * wx + k;
    if (gx >= R && gx < p.w - KSZ + R) xmask |= 0xffu << (8 * k);
  }
  uint32_t kk[KSZ];
#pragma unroll
  for (int j = 0; j < KSZ; j++) kk[j] = p.blur_k[j];
  uint32_t he[KSZ], ho[KSZ];  // even / odd bytes of the row-filtered words of the last KSZ rows
#pragma unroll
  for (int j = 0; j < KSZ; j++) he[j] = ho[j] = 0;
  auto load_row = [&](int t, uint32_t &c, uint32_t &e) {  // t = row of the strip's input window
    const int gy = gy0 - R + t;
    c = 0; e = 0;
    if (t < kBlurRows + 2 * R && gy >= 0 && gy < p.h) {
      const uint32_t *row = src + static_cast<size_t>(gy) * ww;
      if (in_x) c = __ldg(row + wx);
      if (has_ex) e = __ldg(row + ex);
    }
  };
  // rows are fetched kBlurAhead at a time, one group ahead of the filter: a warp keeps 2 * kBlurAhead rows (1 KB) in flight
  constexpr int kTrips = (kBlurRows + 2 * R + kBlurAhead - 1) / kBlurAhead;
  uint32_t nc[kBlurAhead], ne[kBlurAhead];
#pragma unroll
  for (int u = 0; u < kBlurAhead; u++) load_row(u, nc[u], ne[u]);
  uint32_t tmn = 0xffffffffu, tmx = 0;  // byte-wise min / max of this lane's word over the rows of a 4x4 tile
  uint8_t *mm_raw = p.minmax_raw + frame * static_cast<size_t>(p.tiles_x) * p.tiles_y * 2;
  for (int trip = 0; trip < kTrips; trip++) {
    uint32_t cc[kBlurAhead], ce[kBlurAhead];
#pragma unroll
    for (int u = 0; u < kBlurAhead; u++) {
      cc[u] = nc[u];
      ce[u] = ne[u];
    }
#pragma unroll
    for (int u = 0; u < kBlurAhead; u++) load_row((trip + 1) * kBlurAhead + u, nc[u], ne[u]);
#pragma unroll
    for (int u = 0; u < kBlurAhead; u++) {
      const int t = trip * kBlurAhead + u;
      const uint32_t center = cc[u], extra = ce[u];
      uint32_t left = __shfl_up_sync(0xffffffffu, center, 1), right = __shfl_down_sync(0xffffffffu, center, 1);
      if (lane == 0) left = extra;
      if (lane == 31) right = extra;
      uint32_t ae = 0, ao = 0;
#pragma unroll
      for (int j = 0; j < KSZ; j++) {
        const int o = j - R;  // byte k of sw = pixel 4 wx + k + o
        const uint32_t sw = o == 0 ? center : (o > 0 ? __funnelshift_r(center, right, 8 * o) : __funnelshift_r(left, center, 32 + 8 * o));
        ae += kk[j] * (sw & 0x00ff00ffu);
        ao += kk[j] * ((sw >> 8) & 0x00ff00ffu);
      }
      uint32_t hw = ((ae >> 8) & 0x00ff00ffu) | (ao & 0xff00ff00u);
      hw = (hw & xmask) | (center & ~xmask);
#pragma unroll
      for (int j = 0; j + 1 < KSZ; j++) {
        he[j] = he[j + 1];
        ho[j] = ho[j + 1];
      }
      he[KSZ - 1] = hw & 0x00ff00ffu;
      ho[KSZ - 1] = (hw >> 8) & 0x00ff00ffu;
      const int oy = gy0 + t - 2 * R;  // the row in the middle of the window
      if (t >= 2 * R && t < kBlurRows + 2 * R && oy < p.h && in_x) {
        uint32_t out = he[R] | (ho[R] << 8);
        if (oy >= R && oy < p.h - KSZ + R) {
          uint32_t ve = 0, vo = 0;
#pragma unroll
          for (int j = 0; j < KSZ; j++) {
            ve += kk[j] * he[j];
            vo += kk[j] * ho[j];
          }
          out = ((ve >> 8) & 0x00ff00ffu) | (vo & 0xff00ff00u);
        }
        if (p.sharpen) {
          const uint32_t orig = __ldg(src + static_cast<size_t>(oy) * ww + wx);
          uint32_t o = 0;
#pragma unroll
          for (int px = 0; px < 4; px++) {
            int sv = 2 * static_cast<int>((orig >> (8 * px)) & 0xff) - static_cast<int>((out >> (8 * px)) & 0xff);
            sv = max(0, min(255, sv));
            o |= static_cast<uint32_t>(sv) << (8 * px);
          }
          out = o;
        }
        dst[static_cast<size_t>(oy) * ww + wx] = out;
        // 4x4 tile min/max (threshold.cu:60-80; k_tile_minmax's job): a word is one row of a tile, strips start on tile rows
        tmn = __vminu4(tmn, out);
        tmx = __vmaxu4(tmx, out);
        if ((oy & 3) == 3) {
          tmn = __vminu4(tmn, tmn >> 16); tmn = __vminu4(tmn, tmn >> 8);
          tmx = __vmaxu4(tmx, tmx >> 16); tmx = __vmaxu4(tmx, tmx >> 8);
          *reinterpret_cast<uchar2 *>(mm_raw + (static_cast<size_t>(oy >> 2) * p.tiles_x + wx) * 2) = make_uchar2(tmn & 0xff, tmx & 0xff);
          tmn = 0xffffffffu;
          tmx = 0;
        }
      }
    }
  }
}

// 4x4 tile min/max of the quad image (threshold.cu:60-80).  One thread per tile.
__global__ void __launch_bounds__(128) k_tile_minmax(FrameParams p) {
  const int tx = blockIdx.x * blockDim.x + threadIdx.x;
  const int ty = blockIdx.y;
  const int frame = blockIdx.z;
  if (tx >= p.tiles_x) return;
  const size_t n = static_cast<size_t>(p.w) * p.h;
  const uint8_t *quad = p.quad + frame * n;
  uint32_t mn = 0xffffffffu, mx = 0;
#pragma unroll
  for (int r = 0; r < 4; r++) {
    const uint32_t d = *reinterpret_cast<const uint32_t *>(quad + (static_cast<size_t>(ty) * 4 + r) * p.w + static_cast<size_t>(tx) * 4);
    mn = __vminu4(mn, d);
    mx = __vmaxu4(mx, d);
  }
  mn = __vminu4(mn, mn >> 16);
  mn = __vminu4(mn, mn >> 8);
  mx = __vmaxu4(mx, mx >> 16);
  mx = __vmaxu4(mx, mx >> 8);
  uint8_t *mm = p.minmax_raw + (frame * static_cast<size_t>(p.tiles_x) * p.tiles_y + static_cast<size_t>(ty) * p.tiles_x + tx) * 2;
  *reinterpret_cast<uchar2 *>(mm) = make_uchar2(mn & 0xff, mx & 0xff);
}

// ---------------------------------------------------------------------------------------------
// Connected components.  255 is 8-connected, 0 is 4-connected, 127 joins nothing.
// Label of a component = its smallest pixel index (roots are kept minimal by atomicMin
// links), size[root] = pixel count.
//
// A label word carries its pixel's colour class in bits [30:29] from the moment it is written (0 black,
// 1 white, 2 gray): both ends of every union have the same colour, so the bits ride through find / atomicMin
// unchanged, and the later kernels read labels only -- never the thresholded image or, per pixel, the sizes.
// k_ccl_final adds bit 28 = "component has at least 25 pixels".  [27:0] is the label proper.
// ---------------------------------------------------------------------------------------------
constexpr int kCclTW = 32;  // tile width: one 32-bit run mask per row and colour
constexpr int kCclTH = 64;  // tile height
constexpr int kCclThreads = 128;
static_assert(kCclThreads == 2 * kCclTH, "one thread per (row, colour)");
static_assert(kCclThreads == (kCclTW / 4) * (kCclTH / 4), "one thread per 4x4 threshold tile of the CCL tile");

// Find with path halving.  Parent links only ever move to an ancestor (a smaller index of the same
// component), so the plain stores are safe next to the atomicMin links of concurrent unions.  On
// thresholded noise the white (8-connected) pixels percolate into one tile-spanning component;
// without halving its parent chains grow to hundreds of dependent shared-memory hops.
__device__ __forceinline__ uint32_t sfind(uint32_t *par, uint32_t a) {
  uint32_t q = par[a];
  while (q != a) {
    const uint32_t qq = par[q];
    if (qq != q) par[a] = qq;
    a = q;
    q = qq;
  }
  return a;
}

// Unites the trees of a and b (any nodes of them) and returns the root of the result as seen by this thread --
// a valid starting point for the caller's next union on the same run.
__device__ __forceinline__ uint32_t sunite(uint32_t *par, uint32_t a, uint32_t b) {
  while (true) {
    a = sfind(par, a);
    b = sfind(par, b);
    if (a == b) return a;
    if (a < b) {
      const uint32_t t = a;
      a = b;
      b = t;
    }
    const uint32_t old = atomicMin(&par[a], b);
    if (old == a) return b;
    a = old;
  }
}

// Phase (C) of k_ccl_local keeps a root's counters in the upper bits of its own parent word (no second array: 9 KB of
// shared memory per CTA instead of 17, 16 CTAs per SM instead of 12): finds mask the index, and only non-roots -- whose
// words carry no counters -- are ever re-pointed.
constexpr int kParBits = 11;                    // a tile has 2^11 pixels
constexpr uint32_t kParMask = (1u << kParBits) - 1u;
constexpr int kParTouchShift = kParBits + 12;   // the pixel count takes 12 bits (<= 2048)
static_assert(kCclTW * kCclTH == (1 << kParBits), "tile size");
__device__ __forceinline__ uint32_t sfind_counted(uint32_t *par, uint32_t a) {
  uint32_t q = par[a] & kParMask;
  while (q != a) {
    const uint32_t qq = par[q] & kParMask;
    if (qq != q) par[a] = qq;
    a = q;
    q = qq;
  }
  return a;
}

constexpr uint32_t kLabelMask = 0x0fffffffu;   // [27:0] label
constexpr uint32_t kLabelBig = 1u << 28;       // component has >= kMinBlobPixels pixels (set by k_ccl_final)
constexpr int kColourShift = 29;               // [30:29] 0 black, 1 white, 2 gray
constexpr uint32_t kColourGray = 2u << kColourShift;
// tile roots that touch their tile's border (the only ones a cross-tile merge can dethrone): at most one per border pixel
constexpr uint32_t kCclRootCap = 2 * kCclTW + 2 * kCclTH;

// K2+K3: adaptive threshold (threshold.cu:84-147) fused with the tile-local labelling
// (labeling_allegretti_2019_BKE.cu:114-300).  One CTA = a 32x64 tile of the quad image = 8x16 threshold tiles.
//   (T) thread = one 4x4 threshold tile: 3x3 dilation of the raw tile min/max (edge tiles skip missing
//       neighbours), threshold value into shared memory;
//   (A) thread = half a row (one 16-byte load): byte-wise compares (__vcmpgtu4) give the thresholded words, stored
//       as they are, and the white / black bits of the row's two 32-bit run masks -- the labelling never reads the
//       thresholded image back;
//   (B) union-find on RUNS: nodes are the first pixels of the horizontal runs; one thread per (row, colour) walks
//       the runs of its mask with ffs/clz and unites each with the runs it touches in the row above (white:
//       8-connected, i.e. the run dilated by one pixel; black: 4-connected);
//   (C) a second walk compresses every run start to its root and adds the run length to the root's pixel count, kept
//       above the index in the root's own parent word (and above that: how many of the runs touch the tile border);
//   (D) write-out per pixel, 16-byte stores: label = global index of the root of the pixel's run | colour, sizes =
//       count at tile roots, 0 elsewhere; tile roots that touch the border go to the tile's root list, from which
//       k_ccl_handoff moves the counts of merged-away roots to the final roots.
// (tried: a run's first link to the row above as ONE atomicMin on the run's own word -- it still is its own root unless a
//  run below has linked it already, and any smaller index of the other component keeps the forest valid -- instead of two
//  finds and the atomicMin: correct, but the links to non-roots make the later finds longer, 0.269 -> 0.298 ms)
__global__ void __launch_bounds__(kCclThreads, 16) k_ccl_local(FrameParams p) {
  __shared__ uint32_t s_mask[2][kCclTH];  // [0] black, [1] white
  // parent links; from phase (C) on a ROOT's word also carries its counters above the index (kParBits):
  // [10:0] parent | [22:11] pixels of the component (<= 2048) | [30:23] runs of it that touch the tile border (<= 192)
  __shared__ uint32_t s_par[kCclTH * kCclTW];
  __shared__ uint16_t s_thr[kCclTH / 4][kCclTW / 4];  // threshold of the 4x4 tile; 0xffff = flat (all 127)
  __shared__ uint32_t s_roots[kCclRootCap];
  __shared__ uint32_t s_nroots;

  const int frame = blockIdx.z;
  const int x0 = blockIdx.x * kCclTW, y0 = blockIdx.y * kCclTH;
  const size_t n = static_cast<size_t>(p.w) * p.h;
  const uint8_t *quad = p.quad + frame * n;
  uint8_t *th = p.thresh + frame * n;
  uint32_t *labels = p.labels + frame * n;
  uint32_t *sizes = p.sizes + frame * n;
  const int tid = threadIdx.x;

  {  // (T)
    const int tlx = tid & 7, tly = tid >> 3;
    const int tx = (x0 >> 2) + tlx, ty = (y0 >> 2) + tly;
    uint32_t enc = 0xffffu;
    if (tx < p.tiles_x && ty < p.tiles_y) {
      const size_t tiles = static_cast<size_t>(p.tiles_x) * p.tiles_y;
      const uchar2 *raw = reinterpret_cast<const uchar2 *>(p.minmax_raw + frame * tiles * 2);
      int mn = 255, mx = 0;
#pragma unroll
      for (int j = -1; j <= 1; j++) {
        const int ry = ty + j;
        if (ry < 0 || ry >= p.tiles_y) continue;
#pragma unroll
        for (int i = -1; i <= 1; i++) {
          const int rx = tx + i;
          if (rx < 0 || rx >= p.tiles_x) continue;
          const uchar2 m = __ldg(raw + static_cast<size_t>(ry) * p.tiles_x + rx);
          mn = min(mn, static_cast<int>(m.x));
          mx = max(mx, static_cast<int>(m.y));
        }
      }
      if (p.keep_stages) {
        uint8_t *mm = p.minmax + (frame * tiles + static_cast<size_t>(ty) * p.tiles_x + tx) * 2;
        *reinterpret_cast<uchar2 *>(mm) = make_uchar2(mn, mx);
      }
      if ((mx - mn) >= p.min_white_black_diff) enc = static_cast<uint32_t>(mn + (mx - mn) / 2);
    }
    s_thr[tly][tlx] = static_cast<uint16_t>(enc);
    if (tid == 0) s_nroots = 0;
  }
  __syncthreads();

  // (A) thresholded pixels + run masks: thread = half a row (16 pixels: one 16-byte load, one 16-byte store); the
  //     byte-wise compare of each 4-pixel word gives the thresholded word and a nibble of the white / black masks; the
  //     two halves of a row meet with one shuffle.  Pixels outside the image join nothing.
  {
    static_assert(kCclThreads == 2 * kCclTH && kCclTW == 32, "two threads per row");
    const int r = tid >> 1, half = tid & 1;
    const int gy = y0 + r, gx = x0 + 16 * half;
    uint32_t d[4] = {0, 0, 0, 0};
    const bool row_in = gy < p.h;
    const bool vec = row_in && (p.w & 15) == 0 && gx + 16 <= p.w;
    const uint8_t *src = quad + static_cast<size_t>(gy) * p.w + gx;
    if (vec) {
      const uint4 v = __ldg(reinterpret_cast<const uint4 *>(src));
      d[0] = v.x; d[1] = v.y; d[2] = v.z; d[3] = v.w;
    } else if (row_in) {
#pragma unroll
      for (int g = 0; g < 4; g++)
        if (gx + 4 * g < p.w) d[g] = __ldg(reinterpret_cast<const uint32_t *>(src + 4 * g));
    }
    uint32_t o[4], wm16 = 0, bm16 = 0;
#pragma unroll
    for (int g = 0; g < 4; g++) {
      const uint32_t t = s_thr[r >> 2][4 * half + g];
      o[g] = 0x7f7f7f7fu;
      if (t != 0xffffu && row_in && gx + 4 * g < p.w) {
        o[g] = __vcmpgtu4(d[g], t * 0x01010101u);  // 0xff where v > thresh (threshold.cu:138-142)
        const uint32_t wn = ((o[g] & 0x01010101u) * 0x01020408u) >> 24;  // one bit per byte, byte 0 -> bit 0
        wm16 |= wn << (4 * g);
        bm16 |= (wn ^ 0xfu) << (4 * g);
      }
    }
    uint8_t *dst = th + static_cast<size_t>(gy) * p.w + gx;
    if (vec) {
      *reinterpret_cast<uint4 *>(dst) = make_uint4(o[0], o[1], o[2], o[3]);
    } else if (row_in) {
#pragma unroll
      for (int g = 0; g < 4; g++)
        if (gx + 4 * g < p.w) *reinterpret_cast<uint32_t *>(dst + 4 * g) = o[g];
    }
    const uint32_t both = wm16 | (bm16 << 16);
    const uint32_t other = __shfl_xor_sync(0xffffffffu, both, 1);
    if (half == 0) {
      s_mask[1][r] = (both & 0xffffu) | (other << 16);
      s_mask[0][r] = (both >> 16) | (other & 0xffff0000u);
    }
  }
  for (int i = tid; i < kCclTH * kCclTW / 4; i += kCclThreads)
    reinterpret_cast<uint4 *>(s_par)[i] = make_uint4(4 * i, 4 * i + 1, 4 * i + 2, 4 * i + 3);
  __syncthreads();

  // (B) unions with the row above: thread = (row, colour).  Runs come off the mask by carry propagation: adding the
  //     lowest set bit to a mask ripples through the run that starts there, so `m & ~(m + low)` IS that run.
  const int row = tid >> 1, colour = tid & 1;
  const uint32_t mine = s_mask[colour][row];
  if (row > 0) {
    const uint32_t up = s_mask[colour][row - 1];
    uint32_t m = mine;
    while (m) {
      const uint32_t low = m & (0u - m), rest = m + low;
      const uint32_t run = m & ~rest;
      m &= rest;
      const int s = 31 - __clz(static_cast<int>(low));
      uint32_t ov = up & (colour ? (run | (run << 1) | (run >> 1)) : run);
      uint32_t node = row * kCclTW + s;  // replaced by its current root after every union: later finds start there
      while (ov) {
        const uint32_t b = ov & (0u - ov);          // lowest overlapping column
        ov &= ~(up & ~(up + b));                     // ... and the rest of that upper run (from b upwards) is done
        const uint32_t below = ~up & (b - 1u);       // the upper run starts after the last zero below b
        const int us = below ? 32 - __clz(static_cast<int>(below)) : 0;
        node = sunite(s_par, node, (row - 1) * kCclTW + us);
      }
    }
  }
  __syncthreads();

  // (C) compress run starts to their roots; per-root pixel counts and border-touching runs in the roots' parent words
  {
    uint32_t m = mine;
    const bool edge_row = row == 0 || row == kCclTH - 1;
    // consecutive runs of a row often end under the same root (the percolating white component of thresholded noise):
    // their counts are added up in a register and reach the root's word -- a hot address -- in one atomic
    uint32_t acc = 0, acc_root = 0;
    while (m) {
      const uint32_t low = m & (0u - m), rest = m + low;
      const uint32_t run = m & ~rest;
      m &= rest;
      const int s = 31 - __clz(static_cast<int>(low));
      const uint32_t len = static_cast<uint32_t>(__popc(run));
      const uint32_t node = row * kCclTW + s;
      const uint32_t root = sfind_counted(s_par, node);
      if (root != node) s_par[node] = root;  // (a non-root: its word has no counters)
      const uint32_t touches = (edge_row || ((run & 0x80000001u) != 0)) ? (1u << kParTouchShift) : 0u;
      if (root != acc_root && acc) {
        atomicAdd(&s_par[acc_root], acc);
        acc = 0;
      }
      acc_root = root;
      acc += (len << kParBits) | touches;
    }
    if (acc) atomicAdd(&s_par[acc_root], acc);
  }
  __syncthreads();

  // (D) write out, 4 pixels (16 bytes of labels) per thread
  for (int i = tid; i < kCclTH * kCclTW / 4; i += kCclThreads) {
    const int r = i / (kCclTW / 4), xq = (i % (kCclTW / 4)) * 4;
    const int gy = y0 + r, gx = x0 + xq;
    if (gy >= p.h || gx >= p.w) continue;
    const uint32_t wm = s_mask[1][r], bm = s_mask[0][r];
    const size_t g = static_cast<size_t>(gy) * p.w + gx;
    uint32_t lab[4], sz[4];
#pragma unroll
    for (int k = 0; k < 4; k++) {
      const int x = xq + k;
      lab[k] = static_cast<uint32_t>(g + k) | kColourGray;
      sz[k] = 0;
      const bool isw = (wm >> x) & 1u, isb = (bm >> x) & 1u;
      if (isw || isb) {
        const uint32_t below = ~(isw ? wm : bm) & ((1u << x) - 1u);
        const int s = below ? 32 - __clz(static_cast<int>(below)) : 0;
        const uint32_t word = s_par[r * kCclTW + s];
        const uint32_t root = word & kParMask;
        lab[k] = static_cast<uint32_t>((y0 + (root / kCclTW)) * p.w + x0 + (root % kCclTW)) | (isw ? 1u << kColourShift : 0u);
        if (root == static_cast<uint32_t>(r * kCclTW + x)) {  // the pixel is its run's start and the root: `word` is the root's own
          sz[k] = (word >> kParBits) & 0xfffu;
          if (word >> kParTouchShift) s_roots[atomicAdd(&s_nroots, 1u)] = static_cast<uint32_t>(g + k);
        }
      }
    }
    *reinterpret_cast<uint4 *>(labels + g) = make_uint4(lab[0], lab[1], lab[2], lab[3]);
    *reinterpret_cast<uint4 *>(sizes + g) = make_uint4(sz[0], sz[1], sz[2], sz[3]);
  }
  __syncthreads();
  {
    const uint32_t nr = s_nroots;
    const size_t tile = (static_cast<size_t>(frame) * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x;
    uint32_t *list = p.tile_roots + tile * kCclRootCap;
    for (uint32_t i = tid; i < nr; i += kCclThreads) list[i] = s_roots[i];
    if (tid == 0) p.tile_nroots[tile] = nr;
  }
}

// Global find on label words: the index is [27:0], the colour bits travel along (equal at both ends of a link).
__device__ __forceinline__ uint32_t gfind(const uint32_t *par, uint32_t a) {
  uint32_t q = __ldcg(par + (a & kLabelMask));
  while (q != a) {
    a = q;
    q = __ldcg(par + (a & kLabelMask));
  }
  return a;
}

// The same with path halving: every other node on the way is re-pointed at its grandparent.  The plain stores are
// safe next to concurrent atomicMin links for the reason given at sfind.  Worth it only when the chains are walked
// on the critical path of a single frame (a component that spans many tiles is a chain of tile roots): in batches the
// extra stores cost more than the shorter chains save (measured in round 1).
__device__ __forceinline__ uint32_t gfind_halving(uint32_t *par, uint32_t a) {
  uint32_t q = __ldcg(par + (a & kLabelMask));
  while (q != a) {
    const uint32_t qq = __ldcg(par + (q & kLabelMask));
    if (qq != q) par[a & kLabelMask] = qq;
    a = q;
    q = qq;
  }
  return a;
}

template <bool HALVING>
__device__ __forceinline__ void gunite(uint32_t *par, uint32_t a, uint32_t b) {
  while (true) {
    a = HALVING ? gfind_halving(par, a) : gfind(par, a);
    b = HALVING ? gfind_halving(par, b) : gfind(par, b);
    if (a == b) return;
    if (a < b) {
      const uint32_t t = a;
      a = b;
      b = t;
    }
    const uint32_t old = atomicMin(par + (a & kLabelMask), b);
    if (old == a) return;
    a = old;
  }
}

// K4: unions across tile borders.  Work items per tile: its top row (TW), left column (TH),
// right column (TH, for the up-right diagonal).  One thread per item collects up to three
// neighbour pairs (colour from the label words themselves); inside a warp, pairs that join the same two
// tile-local trees (equal raw labels on both sides -- on thresholded noise the same giant component shows up at
// every other border pixel) are deduplicated with __match_any_sync, so only one lane walks the parent chains.
constexpr int kCclMergeThreads = ((kCclTW + 2 * kCclTH + 31) / 32) * 32;
template <bool HALVING>
__global__ void __launch_bounds__(kCclMergeThreads) k_ccl_merge(FrameParams p) {
  const int frame = blockIdx.z;
  const int x0 = blockIdx.x * kCclTW, y0 = blockIdx.y * kCclTH;
  const size_t n = static_cast<size_t>(p.w) * p.h;
  uint32_t *labels = p.labels + frame * n;
  const int t = threadIdx.x, lane = t & 31;
  int x = 0, y = 0;
  int kind = 3;  // 0 top row, 1 left column, 2 right column, 3 idle
  if (t < kCclTW) {
    kind = 0; x = x0 + t; y = y0;
  } else if (t < kCclTW + kCclTH) {
    kind = 1; x = x0; y = y0 + (t - kCclTW);
  } else if (t < kCclTW + 2 * kCclTH) {
    kind = 2; x = x0 + kCclTW - 1; y = y0 + (t - kCclTW - kCclTH);
  }
  uint32_t other[3];  // neighbour pixel of each candidate pair, 0xffffffff = none
  other[0] = other[1] = other[2] = 0xffffffffu;
  uint32_t i = 0;
  const bool live = kind < 3 && x < p.w && y < p.h;
  if (live) i = static_cast<uint32_t>(y * p.w + x);
  const uint32_t mine = __ldcg(labels + i);
  const uint32_t colour = mine >> kColourShift;  // 0 black, 1 white, 2 gray
  // (fetching the diagonal neighbours from the geometry alone, side by side with this pixel's word instead of after its
  //  colour is known, was measured: one round trip less per chain, but a third more loads -- 0.079 -> 0.086 ms)
  if (live && colour != 2) {
    if (kind == 0) {
      if (y > 0) {  // every "up" neighbour is in another tile
        other[0] = i - p.w;
        if (colour == 1) {
          if (x > 0) other[1] = i - p.w - 1;
          if (x + 1 < p.w) other[2] = i - p.w + 1;
        }
      }
    } else if (kind == 1) {
      if (x > 0) {
        other[0] = i - 1;
        // up-left lies in the left tile; rows at the tile top were handled by kind 0
        if (colour == 1 && y > y0) other[1] = i - p.w - 1;
      }
    } else {
      if (colour == 1 && y > y0 && x + 1 < p.w) other[0] = i - p.w + 1;
    }
  }
  uint32_t theirs[3];
#pragma unroll
  for (int k = 0; k < 3; k++) theirs[k] = other[k] != 0xffffffffu ? __ldcg(labels + other[k]) : 0xffffffffu;
#pragma unroll
  for (int k = 0; k < 3; k++) {
    const bool has = other[k] != 0xffffffffu && (theirs[k] >> kColourShift) == colour;
    const uint32_t active = __ballot_sync(0xffffffffu, has);
    if (!has) continue;
    const unsigned long long key = (static_cast<unsigned long long>(min(mine, theirs[k])) << 32) | max(mine, theirs[k]);
    const uint32_t group = __match_any_sync(active, key);
    if (lane == __ffs(group) - 1 && mine != theirs[k]) gunite<HALVING>(labels, mine, theirs[k]);
  }
}

// K4b: tile roots that a cross-tile merge dethroned hand their pixel count to the final root.  Only roots whose
// tile-local component touches the tile border can be affected, and k_ccl_local listed exactly those: one warp
// per tile walks its list (the reference scans every pixel for this, labeling_allegretti_2019_BKE.cu:340-462).
// (two warps per tile, so that more of a list's dependent chains are in flight at once, measured no faster: 0.034 vs 0.033 ms)
template <int TPT>  // threads per tile
__global__ void __launch_bounds__(256) k_ccl_handoff(FrameParams p, uint32_t tiles_per_frame) {
  const int frame = blockIdx.y;
  const size_t n = static_cast<size_t>(p.w) * p.h;
  const uint32_t *labels = p.labels + frame * n;
  uint32_t *sizes = p.sizes + frame * n;
  const uint32_t tile = blockIdx.x * (256 / TPT) + (threadIdx.x / TPT);
  if (tile >= tiles_per_frame) return;
  const size_t t = static_cast<size_t>(frame) * tiles_per_frame + tile;
  const uint32_t nr = p.tile_nroots[t];
  const uint32_t *list = p.tile_roots + t * kCclRootCap;
  for (uint32_t e = threadIdx.x % TPT; e < nr; e += TPT) {
    const uint32_t self = list[e];
    const uint32_t me = __ldcg(labels + self);
    const uint32_t mine = sizes[self];  // (fetched next to the label, not after the chain)
    if ((me & kLabelMask) == self) continue;  // still a root
    const uint32_t root = gfind(labels, me) & kLabelMask;
    atomicAdd(sizes + root, mine);
    sizes[self] = 0;
  }
}

// K5: every pixel gets its final label word: root | colour | "component has at least 25 pixels" (sizes are final
// after k_ccl_handoff).  One CTA per CCL tile: after k_ccl_local every pixel of a tile points at one of the tile's own
// roots, so only those (a few hundred per 2048 pixels) are chased through the merged trees -- once each, into a
// shared-memory table indexed by the root's position in the tile -- and every pixel then takes its word from the
// table.  16 bytes of labels in, 16 bytes out per thread and pass; the dependent global accesses (parent chain, size
// of the final root) happen once per tile root instead of once per pixel.
constexpr int kFinThreads = 256;
constexpr int kFinPasses = kCclTW * kCclTH / 4 / kFinThreads;
constexpr uint32_t kFinUnused = 0xffffffffu, kFinNeeded = 0xfffffffeu;
// (8 CTAs per SM caps it at 32 registers; uncapped it ran at 6 CTAs per SM: 0.111 against 0.097 ms per 128 config-2 frames)
__global__ void __launch_bounds__(kFinThreads, 8) k_ccl_final(FrameParams p) {
  __shared__ uint32_t s_out[kCclTW * kCclTH];
  __shared__ uint16_t s_list[kCclTW * kCclTH];
  __shared__ uint32_t s_nlist;
  const int frame = blockIdx.z;
  const int x0 = blockIdx.x * kCclTW, y0 = blockIdx.y * kCclTH;
  const size_t n = static_cast<size_t>(p.w) * p.h;
  uint32_t *labels = p.labels + frame * n;
  const uint32_t *sizes = p.sizes + frame * n;
  const int tid = threadIdx.x;
  if (tid == 0) s_nlist = 0;
  const uint32_t origin = static_cast<uint32_t>(y0) * p.w + x0;
  for (int i = tid; i < kCclTW * kCclTH / 4; i += kFinThreads)
    reinterpret_cast<uint4 *>(s_out)[i] = make_uint4(kFinUnused, kFinUnused, kFinUnused, kFinUnused);
  uint32_t lab[kFinPasses][4], pos[kFinPasses][4];
#pragma unroll
  for (int k = 0; k < kFinPasses; k++) {
    const int i = tid + k * kFinThreads;
    const int r = i / (kCclTW / 4), xq = (i % (kCclTW / 4)) * 4;
    const int gy = y0 + r, gx = x0 + xq;
    uint4 l = make_uint4(kColourGray, kColourGray, kColourGray, kColourGray);
    if (gy < p.h && gx < p.w) l = __ldcg(reinterpret_cast<const uint4 *>(labels + static_cast<size_t>(gy) * p.w + gx));
    lab[k][0] = l.x; lab[k][1] = l.y; lab[k][2] = l.z; lab[k][3] = l.w;
  }
  __syncthreads();
  // (1) which positions of the tile are roots some pixel points at
#pragma unroll
  for (int k = 0; k < kFinPasses; k++) {
#pragma unroll
    for (int q = 0; q < 4; q++) {
      pos[k][q] = kFinUnused;
      if ((lab[k][q] >> kColourShift) == 2) continue;  // 127-pixels: own index, never large enough
      // position in the tile of the root this pixel points at.  A tile root that a cross-tile merge dethroned
      // points OUT of the tile (at its new parent): it is resolved from its own position.
      const uint32_t delta = (lab[k][q] & kLabelMask) - origin;
      const uint32_t dy = __umulhi(delta, p.inv_w);  // delta / w: exact below 2^20, and >= kCclTH beyond (or on wrap-around)
      const uint32_t dx = delta - dy * p.w;
      const int i = tid + k * kFinThreads;
      const uint32_t own = static_cast<uint32_t>(i / (kCclTW / 4)) * kCclTW + (i % (kCclTW / 4)) * 4 + q;
      pos[k][q] = (dy < kCclTH && dx < kCclTW) ? dy * kCclTW + dx : own;
      s_out[pos[k][q]] = kFinNeeded;
    }
  }
  __syncthreads();
  // (2) resolve them: final root of the merged tree, size of that root.  The needed positions are first compacted
  //     into a list, so that the dependent global accesses of all of them are in flight side by side (one per thread)
  //     instead of one after the other in the threads that happen to own several.
  for (int i = tid; i < kCclTW * kCclTH; i += kFinThreads)
    if (s_out[i] == kFinNeeded) s_list[atomicAdd(&s_nlist, 1u)] = static_cast<uint16_t>(i);
  __syncthreads();
  const uint32_t nlist = s_nlist;
  for (uint32_t u = tid; u < nlist; u += kFinThreads) {
    const int i = s_list[u];
    const uint32_t self = origin + static_cast<uint32_t>(i / kCclTW) * p.w + (i % kCclTW);
    // (loading the root's own size side by side with its cell, on the guess that it was never dethroned, was
    //  measured: the extra gathers cost more than the shorter chains save -- 0.149 -> 0.167 ms per 128 frames)
    const uint32_t root = gfind(labels, __ldcg(labels + self)) & ~kLabelBig;
    const uint32_t size = __ldg(sizes + (root & kLabelMask));
    s_out[i] = root | (size >= kMinBlobPixels ? kLabelBig : 0u);
  }
  __syncthreads();
  // (3) every pixel takes the word of its tile root
#pragma unroll
  for (int k = 0; k < kFinPasses; k++) {
    const int i = tid + k * kFinThreads;
    const int r = i / (kCclTW / 4), xq = (i % (kCclTW / 4)) * 4;
    const int gy = y0 + r, gx = x0 + xq;
    if (gy >= p.h || gx >= p.w) continue;
    uint32_t o[4];
#pragma unroll
    for (int q = 0; q < 4; q++) o[q] = pos[k][q] == kFinUnused ? lab[k][q] : s_out[pos[k][q]];
    *reinterpret_cast<uint4 *>(labels + static_cast<size_t>(gy) * p.w + gx) = make_uint4(o[0], o[1], o[2], o[3]);
  }
}

// ---------------------------------------------------------------------------------------------
// K6: boundary points, grouped by blob pair.
//
// One CTA = one 64x8 pixel tile (halo staged in shared memory as label | big | colour).
//   (1) per pixel: which of the 4 directions emit a point (apriltag_gpu.cu:276-357); the points
//       are compacted into a shared-memory list, so everything after this runs with full warps;
//   (2) per point: blob-pair key -> entry of a CTA-local hash table, local rank by one
//       shared-memory atomicAdd on the entry's count;
//   (3) per local entry: ONE find-or-claim in the frame's global blob-pair hash and ONE global
//       atomicAdd of the entry's count, which returns the base rank of this tile's points;
//   (4) per point: 8-byte record (slot, rank, x, y, dir, polarity), coalesced stores.
// The reference writes a dense 32-byte-per-pixel array, compacts it and radix-sorts it by blob
// pair (C1, C2); extents (C3) are computed per blob by the fit kernels, where a whole blob sits
// in one warp / CTA and the reductions are shuffles instead of atomics.
// ---------------------------------------------------------------------------------------------
constexpr int kBpTW = 64;               // tile width: one 64-bit emission mask per (row, direction)
constexpr uint32_t kBpMaxProbe = 48;    // longer probe sequences take the direct-to-global path
constexpr uint32_t kBpDirect = 0xffffffffu;

__device__ __forceinline__ uint32_t hash_pair(uint32_t a, uint32_t b) {
  uint32_t h = a * 0x9E3779B1u ^ (b * 0x85EBCA77u + 0x165667B1u);
  h ^= h >> 15;
  h *= 0x2C1B3C6Du;
  h ^= h >> 13;
  return h;
}

// Finds or claims the slot of blob pair `key`; returns kInvalidSlot on a full table.
__device__ uint32_t hash_insert(const FrameParams &p, unsigned long long *keys, unsigned long long key, uint32_t rep0, uint32_t rep1,
                                Counters *ctr, uint32_t *occupied) {
  uint32_t slot = hash_pair(rep0, rep1) & (p.hash_cap - 1);
  for (uint32_t probe = 0; probe < p.hash_cap; probe++) {
    // compare-and-swap first: one L2 round trip whether the key is already there or the slot gets claimed
    const unsigned long long cur = atomicCAS(keys + slot, kEmptyKey, key);
    if (cur == key) return slot;
    if (cur == kEmptyKey) {  // we claimed it: list the slot so k_select never scans the whole table
      occupied[atomicAdd(&ctr->num_occupied, 1u)] = slot;
      return slot;
    }
    slot = (slot + 1) & (p.hash_cap - 1);
  }
  atomicOr(&ctr->status, B200TAG_ST_HASH_OVERFLOW);
  return kInvalidSlot;
}

// staged cell = label word: [27:0] label | [28] big enough | [30:29] colour class (0 black, 1 white, 2 gray)
constexpr int kBpTH = 8;                 // tile height; 16 threads per row
constexpr int kBpThreads = kBpTH * 16;
// kBpMaxPts = points of the tile that phases (2)-(4) take in one go.  A tile can emit up to four points per pixel,
// thresholded sensor noise emits 0.75, long one-pixel stripes 2: the list buffers hold 2 points per pixel and a tile with
// more goes through (2)-(4) in several rounds, each with a fresh CTA-local table (ranks stay consistent: every round adds
// its counts to the global table before its records are written).  Half the list memory = 12 instead of 9 CTAs per SM.
constexpr int kBpMaxPts = 1024;
static_assert(kBpMaxPts <= kBpTW * kBpTH * 4 && kBpMaxPts % 32 == 0, "list capacity");
constexpr int kBpLHBits = 8;
constexpr uint32_t kBpLH = 1u << kBpLHBits;  // local blob-pair table (power of two, <= 1024: 10-bit entry index in s_loc)
static_assert(kBpLH <= 1024, "local table size");
// SMALL_ROUNDS: the test variant that takes 96 points per round (B200TAG_TEST_SMALL_CHUNKS), its own instantiation so
// that the production kernel compares against a compile-time capacity.
template <bool SMALL_ROUNDS>
__global__ void __launch_bounds__(kBpThreads) k_boundary(FrameParams p) {
  __shared__ uint32_t s_cell[kBpTH + 1][kBpTW + 2];
  __shared__ uint16_t s_pts[kBpMaxPts];             // [12:3] pixel of the tile | [2:1] dir | [0] black_to_white
  __shared__ uint32_t s_loc[kBpMaxPts];             // [9:0] local entry | [31:10] rank among the tile's points of that entry
  __shared__ __align__(16) unsigned long long s_lkey[kBpLH];  // blob-pair key; after (3): the global slot
  __shared__ __align__(16) uint32_t s_lcnt[kBpLH];            // points of the entry in this tile; after (3): base rank
  __shared__ uint16_t s_used[kBpLH];                // entries in use, in claim order: (3) runs over these, densely
  __shared__ uint32_t s_nused;
  __shared__ uint32_t s_npts, s_gbase;
  __shared__ uint32_t s_rowm[kBpTH + 1][3][2];      // white / black / big masks of a staged row, two 32-bit halves
  __shared__ uint8_t s_halo[kBpTH + 1][2];          // the same three bits for the left / right halo column
  __shared__ unsigned long long s_emit[kBpTH][4], s_b2w[kBpTH][4];
  __shared__ uint32_t s_ebase[kBpTH][4];
  const int frame = blockIdx.z;
  const int x0 = blockIdx.x * kBpTW, y0 = blockIdx.y * kBpTH;
  const size_t n = static_cast<size_t>(p.w) * p.h;
  const uint32_t *labels = p.labels + frame * n;
  Counters *ctr = p.counters + frame;
  uint64_t *points = p.points + static_cast<size_t>(frame) * p.point_cap;
  const size_t hoff = static_cast<size_t>(frame) * p.hash_cap;
  unsigned long long *h_key = p.h_key + hoff;
  uint32_t *h_count = p.h_count + hoff;
  uint32_t *occupied = p.occupied + hoff;
  const int tid = threadIdx.x, lane = tid & 31;

  auto clear_table = [&]() {  // 16-byte stores
    static_assert(kEmptyKey == 0xFFFFFFFFFFFFFFFFull, "all ones");
    for (int i = tid; i < static_cast<int>(kBpLH / 2); i += kBpThreads)
      reinterpret_cast<uint4 *>(s_lkey)[i] = make_uint4(0xffffffffu, 0xffffffffu, 0xffffffffu, 0xffffffffu);
    for (int i = tid; i < static_cast<int>(kBpLH / 4); i += kBpThreads) reinterpret_cast<uint4 *>(s_lcnt)[i] = make_uint4(0, 0, 0, 0);
    if (tid == 0) s_nused = 0;
  };
  clear_table();
  // halo tile: the label words already are the cells (k_ccl_final); outside the image = gray.  A warp stages whole rows
  // (two coalesced 128-byte loads + the two halo cells), so the row masks of (1) -- three 64-bit masks per staged row:
  // white, black, component big enough, plus the same three bits for the two halo columns -- come from ballots over the
  // words it still holds in registers.
  {
    constexpr int kWarps = kBpThreads / 32;
    constexpr int kRowsPer = (kBpTH + 1 + kWarps - 1) / kWarps;
    const int wrp = tid >> 5;
    uint32_t c0[kRowsPer], c1[kRowsPer], ch[kRowsPer];
#pragma unroll
    for (int k = 0; k < kRowsPer; k++) {
      const int r = wrp + k * kWarps, gy = y0 + r;
      c0[k] = c1[k] = ch[k] = kColourGray;
      if (r <= kBpTH && gy < p.h) {
        const uint32_t *row = labels + static_cast<size_t>(gy) * p.w;
        const int gx0 = x0 + lane, gx1 = x0 + 32 + lane;
        const int gxh = lane == 0 ? x0 - 1 : x0 + kBpTW;  // lanes 0 / 1: left / right halo column
        if (gx0 < p.w) c0[k] = __ldg(row + gx0);
        if (gx1 < p.w) c1[k] = __ldg(row + gx1);
        if (lane < 2 && gxh >= 0 && gxh < p.w) ch[k] = __ldg(row + gxh);
      }
    }
#pragma unroll
    for (int k = 0; k < kRowsPer; k++) {
      const int r = wrp + k * kWarps;
      if (r > kBpTH) continue;  // (warp-uniform)
      s_cell[r][1 + lane] = c0[k];
      s_cell[r][33 + lane] = c1[k];
      if (lane < 2) {  // halo columns: bit 0 white, 1 black, 2 big
        s_cell[r][lane ? kBpTW + 1 : 0] = ch[k];
        const uint32_t col = ch[k] >> 29;
        s_halo[r][lane] = static_cast<uint8_t>((col == 1 ? 1u : 0u) | (col == 0 ? 2u : 0u) | (((ch[k] >> 28) & 1u) << 2));
      }
#pragma unroll
      for (int half = 0; half < 2; half++) {
        const uint32_t c = half ? c1[k] : c0[k];
        const uint32_t col = c >> 29;
        const uint32_t wm = __ballot_sync(0xffffffffu, col == 1), bm = __ballot_sync(0xffffffffu, col == 0);
        const uint32_t gm = __ballot_sync(0xffffffffu, (c >> 28) & 1u);
        if (lane == 0) {
          s_rowm[r][0][half] = wm;
          s_rowm[r][1][half] = bm;
          s_rowm[r][2][half] = gm;
        }
      }
    }
  }
  __syncthreads();

  // (1) which directions emit a point -- on row bit masks: one thread per (row, direction) combines the masks into the
  //     emission mask of apriltag_gpu.cu:276-357 with shifts and ANDs; popcounts give every point its place in the
  //     list without shuffles or atomics.
  if (tid < kBpTH * 4) {
    const int ry = tid >> 2, d = tid & 3;
    const int y = y0 + ry;
    auto row64 = [&](int r, int k) { return (static_cast<unsigned long long>(s_rowm[r][k][1]) << 32) | s_rowm[r][k][0]; };
    unsigned long long emit = 0, b2w = 0;
    if (y >= 1 && y <= p.h - 2) {
      const unsigned long long W0 = row64(ry, 0), B0 = row64(ry, 1), G0 = row64(ry, 2);
      const int rn = ry + dir_dy(d), dx = dir_dx(d);
      unsigned long long W1 = row64(rn, 0), B1 = row64(rn, 1), G1 = row64(rn, 2);
      if (dx > 0) {  // neighbour column x + 1: shift right, the right halo enters at bit 63
        const unsigned long long h = s_halo[rn][1];
        W1 = (W1 >> 1) | ((h & 1ull) << 63); B1 = (B1 >> 1) | (((h >> 1) & 1ull) << 63); G1 = (G1 >> 1) | (((h >> 2) & 1ull) << 63);
      } else if (dx < 0) {  // neighbour column x - 1: shift left, the left halo enters at bit 0
        const unsigned long long h = s_halo[rn][0];
        W1 = (W1 << 1) | (h & 1ull); B1 = (B1 << 1) | ((h >> 1) & 1ull); G1 = (G1 << 1) | ((h >> 2) & 1ull);
      }
      b2w = B0 & W1;                                   // :316
      emit = ((W0 & B1) | b2w) & G0 & G1;              // :284,305,306
      if (d == 3) {  // duplicate suppression, :347-357: left and lower neighbours non-gray, different colours, both big
        const unsigned long long hl = s_halo[ry][0];
        const unsigned long long WL = (W0 << 1) | (hl & 1ull), BL = (B0 << 1) | ((hl >> 1) & 1ull), GL = (G0 << 1) | ((hl >> 2) & 1ull);
        const unsigned long long W2 = row64(ry + 1, 0), B2 = row64(ry + 1, 1), G2 = row64(ry + 1, 2);
        unsigned long long skip = ((WL & B2) | (BL & W2)) & GL & G2;
        if (x0 <= 1 && 1 < x0 + kBpTW) skip &= ~(1ull << (1 - x0));  // x != 1
        emit &= ~skip;
      }
      // interior columns only, :239,276-281
      const int xlo = max(1, x0) - x0, xhi = min(p.w - 2, x0 + kBpTW - 1) - x0;  // inclusive, tile-local
      unsigned long long cols = 0;
      if (xhi >= xlo) cols = (xhi - xlo + 1 >= 64 ? ~0ull : ((1ull << (xhi - xlo + 1)) - 1ull)) << xlo;
      emit &= cols;
    }
    s_emit[ry][d] = emit;
    s_b2w[ry][d] = b2w;
    // exclusive prefix of the popcounts over the 32 (row, direction) words: one warp
    static_assert(kBpTH * 4 == 32, "one warp per (row, direction) word");
    const uint32_t cnt = static_cast<uint32_t>(__popcll(emit));
    uint32_t incl = cnt;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += t;
    }
    s_ebase[ry][d] = incl - cnt;
    if (tid == 31) s_npts = incl;
  }
  __syncthreads();
  const uint32_t npts = s_npts;
  if (npts == 0) return;
  if (tid == 0) s_gbase = atomicAdd(&ctr->num_points, npts);
  constexpr uint32_t cap = SMALL_ROUNDS ? 96u : static_cast<uint32_t>(kBpMaxPts);
  const bool one_round = npts <= cap;  // (CTA-uniform)
  for (uint32_t c0 = 0; c0 < npts; c0 += cap) {  // one round unless the tile has more than kBpMaxPts points
    if (c0 > 0) {
      __syncthreads();  // the previous round's records are written: list and table are free again
      clear_table();
    }
    {  // list entries: one thread per 16-bit quarter of an emission word walks its set bits (3 on average)
      static_assert(kBpThreads == kBpTH * 4 * 4 && kBpTW == 64, "one thread per (row, direction, quarter)");
      const int ry = tid >> 4, d = (tid >> 2) & 3, q = tid & 3;
      const unsigned long long e = s_emit[ry][d];
      uint32_t piece = static_cast<uint32_t>(e >> (16 * q)) & 0xffffu;
      const uint32_t bw = static_cast<uint32_t>(s_b2w[ry][d] >> (16 * q));
      uint32_t pos = s_ebase[ry][d] + __popcll(e & ((1ull << (16 * q)) - 1ull)) - c0;  // (wraps below c0: not in this round)
      const uint32_t head = (static_cast<uint32_t>(ry * kBpTW + 16 * q) << 3) | (d << 1);
      if (one_round) {
        while (piece) {
          const int b = __ffs(static_cast<int>(piece)) - 1;
          piece &= piece - 1;
          s_pts[pos++] = static_cast<uint16_t>(head + (b << 3) + ((bw >> b) & 1u));
        }
      } else {
        while (piece) {
          const int b = __ffs(static_cast<int>(piece)) - 1;
          piece &= piece - 1;
          if (pos < cap) s_pts[pos] = static_cast<uint16_t>(head + (b << 3) + ((bw >> b) & 1u));
          pos++;
        }
      }
    }
    __syncthreads();
    const uint32_t m = min(cap, npts - c0);

    // (2) local blob-pair table: entry + local rank per point
    for (uint32_t i = tid; i < m; i += kBpThreads) {
      const uint32_t e = s_pts[i];
      const uint32_t d = (e >> 1) & 3u, pix = e >> 3;
      const int ry = pix / kBpTW, txp = pix % kBpTW;
      const uint32_t r0 = s_cell[ry][txp + 1] & 0x0fffffffu;
      const uint32_t r1 = s_cell[ry + dir_dy(d)][txp + 1 + dir_dx(d)] & 0x0fffffffu;
      const uint32_t ra = min(r0, r1), rb = max(r0, r1);
      const unsigned long long key = (static_cast<unsigned long long>(ra) << 32) | rb;
      // (the CTA-local table only has to spread the few dozen pairs of one tile: two multiplies, top bits)
      uint32_t h = ((ra * 0x9E3779B1u) ^ (rb * 0x85EBCA77u)) >> (32 - kBpLHBits);
      uint32_t loc = kBpDirect;  // crowded local table (adversarial input): handled in (4)
      const uint32_t max_probe = (p.test_flags & B200TAG_TEST_DIRECT_HASH) ? 0u : kBpMaxProbe;
      for (uint32_t probe = 0; probe < max_probe; probe++) {
        unsigned long long cur = *reinterpret_cast<volatile unsigned long long *>(&s_lkey[h]);
        if (cur == kEmptyKey) {
          cur = atomicCAS(&s_lkey[h], kEmptyKey, key);
          if (cur == kEmptyKey) s_used[atomicAdd(&s_nused, 1u)] = static_cast<uint16_t>(h);  // claimed: list it
        }
        if (cur == key || cur == kEmptyKey) {
          loc = h | (atomicAdd(&s_lcnt[h], 1u) << 10);
          break;
        }
        h = (h + 1) & (kBpLH - 1);
      }
      s_loc[i] = loc;
    }
    __syncthreads();

    // (3) one global find-or-claim and one global count update per local entry
    const uint32_t nused = s_nused;
    for (uint32_t u = tid; u < nused; u += kBpThreads) {
      const uint32_t e = s_used[u];
      const unsigned long long key = s_lkey[e];
      const uint32_t slot = hash_insert(p, h_key, key, static_cast<uint32_t>(key >> 32), static_cast<uint32_t>(key), ctr, occupied);
      s_lkey[e] = slot;
      s_lcnt[e] = slot != kInvalidSlot ? atomicAdd(h_count + slot, s_lcnt[e]) : 0u;
    }
    __syncthreads();

    // (4) point records
    const uint32_t gbase = s_gbase + c0;
    for (uint32_t i = tid; i < m; i += kBpThreads) {
      const uint32_t e = s_pts[i];
      const uint32_t d = (e >> 1) & 3u, pix = e >> 3;
      const int ry = pix / kBpTW, txp = pix % kBpTW;
      const uint32_t loc = s_loc[i];
      uint32_t slot, rank;
      if (loc != kBpDirect) {
        slot = static_cast<uint32_t>(s_lkey[loc & (kBpLH - 1)]);
        rank = s_lcnt[loc & (kBpLH - 1)] + (loc >> 10);
      } else {
        const uint32_t r0 = s_cell[ry][txp + 1] & 0x0fffffffu;
        const uint32_t r1 = s_cell[ry + dir_dy(d)][txp + 1 + dir_dx(d)] & 0x0fffffffu;
        const uint32_t ra = min(r0, r1), rb = max(r0, r1);
        slot = hash_insert(p, h_key, (static_cast<unsigned long long>(ra) << 32) | rb, ra, rb, ctr, occupied);
        rank = slot != kInvalidSlot ? atomicAdd(h_count + slot, 1u) : 0u;
      }
      const uint32_t pos = gbase + i;
      if (pos < p.point_cap) {
        points[pos] = pack_point(slot, rank, static_cast<uint32_t>(x0 + txp), static_cast<uint32_t>(y0 + ry), d, e & 1u);
      } else {
        atomicOr(&ctr->status, B200TAG_ST_POINTS_OVERFLOW);
      }
    }
  }
}

// Resets the blob-pair hash of every frame (first use; afterwards k_select leaves it empty).
__global__ void k_hash_clear(FrameParams p, int frames) {
  const size_t total = static_cast<size_t>(frames) * p.hash_cap;
  for (size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < total; i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    p.h_key[i] = kEmptyKey;
    p.h_count[i] = 0;
  }
}

// ---------------------------------------------------------------------------------------------
// launch helpers
// ---------------------------------------------------------------------------------------------
static inline unsigned cdiv(unsigned a, unsigned b) { return (a + b - 1) / b; }

void launch_frontend(const FrameParams &p, int frames, Launcher &ln) {
  const cudaStream_t s = ln.s;
  const dim3 tgrid(cdiv(p.tiles_x, 128), p.tiles_y, frames);
  if (p.fmt == B200TAG_FMT_YUYV && p.f == 2 && !p.blur_ksz) {
    ln.timed("pre_yuyv_dec2", [&] { k_pre_yuyv_dec2<<<tgrid, 128, 0, s>>>(p); });
  } else if (p.fmt == B200TAG_FMT_BGR8 && p.f == 2 && !p.blur_ksz && (reinterpret_cast<uintptr_t>(p.in) | p.in_stride) % 8 == 0) {
    ln.timed("pre_bgr_dec2", [&] { k_pre_bgr_dec2<<<tgrid, 128, 0, s>>>(p); });
  } else if (p.fmt == B200TAG_FMT_GRAY8 && p.f == 2 && !p.blur_ksz && (reinterpret_cast<uintptr_t>(p.in) | p.in_stride) % 8 == 0) {
    ln.timed("pre_gray_dec2", [&] { k_pre_gray_dec2<<<tgrid, 128, 0, s>>>(p); });
  } else {
    const bool vec_bgr = (p.fmt == B200TAG_FMT_BGR8 && p.f == 1 && (static_cast<size_t>(p.W) * p.H) % 16 == 0 && p.in_stride % 16 == 0);
    if (vec_bgr) {
      const size_t groups = static_cast<size_t>(p.W) * p.H / 16;
      ln.timed("pre_bgr_dec1", [&] { k_pre_bgr_dec1<<<dim3(cdiv(static_cast<unsigned>(groups), 256), frames), 256, 0, s>>>(p); });
    } else {
      ln.timed("pre_generic", [&] { k_pre_generic<<<tgrid, 128, 0, s>>>(p, p.blur_ksz ? 0 : 1); });
    }
    if (p.blur_ksz) {
      const int r = p.blur_ksz >> 1, r4 = (r + 3) & ~3;
      const size_t smem = static_cast<size_t>(kBlurTH + 2 * r) * (kBlurTW + 2 * r4) + static_cast<size_t>(kBlurTH + 2 * r) * kBlurTW;
      const dim3 bgrid(cdiv(p.w, kBlurTW), cdiv(p.h, kBlurTH), frames);
      // (the quad image is word aligned: its width is a multiple of 4 and so is every frame's size)
      const dim3 sgrid(cdiv(p.w / 4, 32), cdiv(p.h, 4 * kBlurRows), frames);
      ln.timed("blur", [&] {
        switch (p.blur_ksz) {
          case 3: k_blur_strip<3><<<sgrid, 128, 0, s>>>(p); break;
          case 5: k_blur_strip<5><<<sgrid, 128, 0, s>>>(p); break;
          case 7: k_blur_strip<7><<<sgrid, 128, 0, s>>>(p); break;
          default: k_blur<<<bgrid, 256, smem, s>>>(p); break;
        }
      });
    }
    const bool minmax_done = p.blur_ksz >= 3 && p.blur_ksz <= 7;  // k_blur_strip writes the tile min/max itself
    if ((p.blur_ksz || vec_bgr) && !minmax_done) ln.timed("tile_minmax", [&] { k_tile_minmax<<<tgrid, 128, 0, s>>>(p); });
  }
  const dim3 cgrid(cdiv(p.w, kCclTW), cdiv(p.h, kCclTH), frames);
  ln.timed("ccl_local", [&] { k_ccl_local<<<cgrid, kCclThreads, 0, s>>>(p); });
  ln.timed("ccl_merge", [&] {
    if (frames <= 4) k_ccl_merge<true><<<cgrid, kCclMergeThreads, 0, s>>>(p);   // single-frame latency: see gfind_halving
    else k_ccl_merge<false><<<cgrid, kCclMergeThreads, 0, s>>>(p);
  });
  ln.timed("ccl_handoff", [&] { k_ccl_handoff<32><<<dim3(cdiv(cgrid.x * cgrid.y, 8), frames), 256, 0, s>>>(p, cgrid.x * cgrid.y); });
  ln.timed("ccl_final", [&] { k_ccl_final<<<cgrid, kFinThreads, 0, s>>>(p); });
  ln.timed("boundary", [&] {
    const dim3 g(cdiv(p.w, kBpTW), cdiv(p.h, kBpTH), frames);
    if (p.test_flags & B200TAG_TEST_SMALL_CHUNKS) k_boundary<true><<<g, kBpThreads, 0, s>>>(p);
    else k_boundary<false><<<g, kBpThreads, 0, s>>>(p);
  });
}

size_t ccl_tiles_per_frame(int w, int h) { return static_cast<size_t>(cdiv(w, kCclTW)) * cdiv(h, kCclTH); }
size_t ccl_root_cap() { return kCclRootCap; }

void launch_hash_clear(const FrameParams &p, int frames, cudaStream_t s) {
  k_hash_clear<<<296, 256, 0, s>>>(p, frames);
}

}  // namespace b200tag
