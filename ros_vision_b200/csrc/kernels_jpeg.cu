// Baseline-JPEG luminance decoder on the GPU (camera wire format, SURVEY section 8 row f2).  The reference leaves MJPG
// decoding to OpenCV on the CPU (src/usb_camera/src/camera_publisher.cpp:198,336) and then converts bgr8 -> YUYV ->
// gray; the detector only ever looks at luminance, so these kernels decode exactly that plane, straight into the
// detector's input staging buffer.  Chrominance blocks are parsed and dropped.
//
// Two paths:
//  * parallel (every well-formed stream): unstuffing (k_jpeg_unstuff*), then the Huffman-coded scan is decoded by one
//    thread per 512-bit subsequence -- streams without restart markers by self-synchronisation (k_jpeg_sync rounds to
//    a proven fixed point, k_jpeg_blockscan, k_jpeg_write; see jpeg_core.h), streams with restart markers one thread
//    per restart interval (k_jpeg_write_rst) --, DC prediction as a scan (k_jpeg_dcscan), and the inverse DCT with
//    eight threads per block (k_jpeg_idct);
//  * sequential (k_jpeg_luma, the fallback for frames the parallel path could not prove): one warp per frame.  All 32
//    lanes run the entropy decoder redundantly on identical state (same instructions, same data: no divergence, no
//    cost over a single thread), which keeps every branch warp-uniform and lets the lanes split the data-parallel
//    parts: byte unstuffing into a shared-memory ring (ballot / popc compaction), the inverse DCT and the pixel stores.
// Both paths, and the host model in jpeg_host.cc, share jpeg_idct8 and produce identical planes.
#include <cuda_runtime.h>

#include <cstdint>

#include "jpeg.h"
#include "jpeg_core.h"
#include "kernels.h"

namespace b200tag {
namespace {

constexpr int kRingBytes = 1024;  // unstuffed entropy-coded bytes staged in shared memory (power of two)
constexpr int kRingWords = kRingBytes / 4;

__constant__ uint8_t c_zigzag[64] = {0,  1,  8,  16, 9,  2,  3,  10, 17, 24, 32, 25, 18, 11, 4,  5,  12, 19, 26, 33, 40, 48,
                                     41, 34, 27, 20, 13, 6,  7,  14, 21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23,
                                     30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63};

struct Shared {
  JpegTables tab;
  JpegFrame frame;
  uint32_t ring[kRingWords];
  float coef[64];  // dequantised coefficients of the current block, natural order
  float tmp[64];
  float quant[64];
  uint8_t zigzag[64];
};

// Input side: raw bytes -> ring of unstuffed bytes (T.81 B.1.1.5: FF 00 stands for a data byte FF; FF followed by
// anything else is a marker and ends the segment).
struct Feeder {
  const uint8_t *src;
  uint32_t gpos, end;   // next raw byte, end of the JPEG
  uint32_t wr;          // bytes written to the ring (monotonic)
  uint32_t prev;        // last raw byte of the previous window (for an FF / 00 pair split across windows)
  bool stopped;         // a marker (or the end of the data) was reached at gpos
};

__device__ __forceinline__ void feed(Feeder &f, uint32_t rd_words, uint8_t *ring_bytes, int lane) {
  // keep the ring topped up: at least kRingBytes - 64 bytes ahead of the reader while input lasts; zero padding after
  // the end of the segment (a well-formed interval never reads it)
  while (f.wr - 4u * rd_words <= static_cast<uint32_t>(kRingBytes - 64)) {
    if (f.stopped) {
      ring_bytes[(f.wr + lane) & (kRingBytes - 1)] = 0;
      f.wr += 32;
      continue;
    }
    const uint32_t idx = f.gpos + lane;
    const uint32_t b = idx < f.end ? f.src[idx] : 0xffu;               // past the end reads as a marker (FF D9)
    uint32_t nb = __shfl_down_sync(0xffffffffu, b, 1);
    if (lane == 31) nb = idx + 1 < f.end ? f.src[idx + 1] : 0xd9u;
    uint32_t pb = __shfl_up_sync(0xffffffffu, b, 1);
    if (lane == 0) pb = f.prev;
    const bool marker = (b == 0xffu && nb != 0u) || idx >= f.end;
    const bool drop = (pb == 0xffu && b == 0u);
    const uint32_t mmask = __ballot_sync(0xffffffffu, marker);
    const int first = mmask ? __ffs(mmask) - 1 : 32;
    const bool keep = lane < first && !drop;
    const uint32_t kmask = __ballot_sync(0xffffffffu, keep);
    if (keep) ring_bytes[(f.wr + __popc(kmask & ((1u << lane) - 1u))) & (kRingBytes - 1)] = static_cast<uint8_t>(b);
    f.wr += __popc(kmask);
    if (first < 32) {
      f.stopped = true;
      f.gpos += first;
    } else {
      f.gpos += 32;
      f.prev = __shfl_sync(0xffffffffu, b, 31);
    }
  }
  __syncwarp();
}

struct BitReader {
  unsigned long long acc;
  int nbits;
  uint32_t rd;  // ring words consumed
};

__device__ __forceinline__ void ensure(BitReader &r, const uint32_t *ring) {
  if (r.nbits <= 32) {
    const uint32_t w = ring[r.rd & (kRingWords - 1)];
    r.acc = (r.acc << 32) | __byte_perm(w, 0, 0x0123);
    r.nbits += 32;
    r.rd++;
  }
}

// F.2.2.3 DECODE: 9-bit lookahead, canonical bounds for longer codes.  Needs nbits >= 16.
__device__ __forceinline__ uint32_t decode_symbol(BitReader &r, const JpegHuff &h) {
  const uint32_t peek = static_cast<uint32_t>(r.acc >> (r.nbits - 16)) & 0xffffu;
  const uint32_t e = h.fast[peek >> (16 - kJpegFastBits)];
  if (e) {
    r.nbits -= static_cast<int>(e >> 8);
    return e & 0xffu;
  }
  int l = kJpegFastBits + 1;
  while (l <= 16 && static_cast<int>(peek >> (16 - l)) > h.maxcode[l]) l++;
  if (l > 16) {  // not a code of this table (corrupt stream)
    r.nbits -= 16;
    return 0;
  }
  r.nbits -= l;
  return h.vals[(h.valoff[l] + static_cast<int>(peek >> (16 - l))) & 0xff];
}

// F.2.2.1 RECEIVE + EXTEND; s <= 11 bits, available after decode_symbol without another refill
__device__ __forceinline__ int receive_extend(BitReader &r, uint32_t s) {
  if (s == 0) return 0;
  const int v = static_cast<int>(static_cast<uint32_t>(r.acc >> (r.nbits - static_cast<int>(s))) & ((1u << s) - 1u));
  r.nbits -= static_cast<int>(s);
  return v < (1 << (s - 1)) ? v - (1 << s) + 1 : v;
}

__global__ void __launch_bounds__(32) k_jpeg_luma(const uint8_t *__restrict__ bits, const JpegFrame *__restrict__ frames,
                                                  const JpegTables *__restrict__ tables, uint8_t *__restrict__ out,
                                                  size_t out_stride, const uint32_t *__restrict__ proven) {
  __shared__ Shared S;
  const int lane = threadIdx.x;
  if (proven && proven[blockIdx.x]) return;  // the parallel kernels decoded this frame
  static_assert(sizeof(JpegFrame) % 4 == 0 && sizeof(JpegTables) % 4 == 0, "copied as words");
  {
    const uint32_t *src = reinterpret_cast<const uint32_t *>(frames + blockIdx.x);
    uint32_t *dst = reinterpret_cast<uint32_t *>(&S.frame);
    for (uint32_t i = lane; i < sizeof(JpegFrame) / 4; i += 32) dst[i] = src[i];
  }
  __syncwarp();
  const JpegFrame *F = &S.frame;
  {
    const uint32_t *src = reinterpret_cast<const uint32_t *>(tables + F->tables);
    uint32_t *dst = reinterpret_cast<uint32_t *>(&S.tab);
    for (uint32_t i = lane; i < sizeof(JpegTables) / 4; i += 32) dst[i] = src[i];
    for (int i = lane; i < 64; i += 32) {
      S.quant[i] = static_cast<float>(F->quant[i]);
      S.zigzag[i] = c_zigzag[i];
    }
  }
  const int width = F->width, height = F->height;
  const int mcus_x = F->mcus_x, nmcu = F->mcus_x * F->mcus_y;
  const int nblocks = F->nblocks, hmax = F->hmax, vmax = F->vmax;
  const int restart = F->restart_interval;
  uint8_t *img = out + static_cast<size_t>(blockIdx.x) * out_stride;
  uint8_t *ring_bytes = reinterpret_cast<uint8_t *>(S.ring);

  Feeder fd;
  fd.src = bits + F->data_off;
  fd.gpos = 0;
  fd.end = F->data_len;
  fd.wr = 0;
  fd.prev = 0x100u;
  fd.stopped = false;
  BitReader br;
  br.acc = 0;
  br.nbits = 0;
  br.rd = 0;
  int pred0 = 0, pred1 = 0, pred2 = 0;  // DC predictors (F.2.1.3.1)
  int until_restart = restart;
  __syncwarp();

  int mx = 0, my = 0;
  for (int m = 0; m < nmcu; m++) {
    if (restart && until_restart == 0) {
      // E.2.4: the interval is followed by an RSTn marker; find it (the feeder normally stopped exactly there), step
      // over it and start the next interval on a byte boundary with zero predictors
      while (!fd.stopped) {
        fd.wr = 4u * br.rd;  // discard
        feed(fd, br.rd, ring_bytes, lane);
        br.rd = fd.wr / 4u;  // (feed only returns with the ring nearly full or the marker found)
      }
      const uint32_t mk = fd.gpos + 1 < fd.end ? fd.src[fd.gpos + 1] : 0xd9u;
      if (fd.gpos < fd.end && mk >= 0xd0u && mk <= 0xd7u) {
        fd.gpos += 2;
        fd.stopped = false;
        fd.prev = 0x100u;
      }
      fd.wr = 0;
      br.rd = 0;
      br.acc = 0;
      br.nbits = 0;
      pred0 = pred1 = pred2 = 0;
      until_restart = restart;
      __syncwarp();
    }
    until_restart--;
    for (int blk = 0; blk < nblocks; blk++) {
      feed(fd, br.rd, ring_bytes, lane);
      const int comp = F->blk_comp[blk];
      const bool luma = comp == 0;
      const JpegHuff &hdc = S.tab.dc[F->comp_dc[comp]];
      const JpegHuff &hac = S.tab.ac[F->comp_ac[comp]];
      if (luma) {
        S.coef[lane] = 0.0f;
        S.coef[lane + 32] = 0.0f;
      }
      __syncwarp();
      ensure(br, S.ring);
      const uint32_t t = decode_symbol(br, hdc) & 15u;
      ensure(br, S.ring);
      const int diff = receive_extend(br, t > 11u ? 11u : t);
      if (comp == 0) pred0 += diff;
      else if (comp == 1) pred1 += diff;
      else pred2 += diff;
      bool any_ac = false;
      if (luma && lane == 0) S.coef[0] = static_cast<float>(pred0) * S.quant[0];
      for (int k = 1; k < 64;) {
        ensure(br, S.ring);
        const uint32_t rs = decode_symbol(br, hac);
        const uint32_t run = rs >> 4, s = rs & 15u;
        if (s == 0) {
          if (run != 15u) break;  // EOB
          k += 16;                // ZRL
          continue;
        }
        k += static_cast<int>(run);
        if (k > 63) break;
        const int v = receive_extend(br, s > 10u ? 10u : s);
        if (luma && lane == 0) {
          const int nat = S.zigzag[k];
          S.coef[nat] = static_cast<float>(v) * S.quant[nat];
        }
        any_ac = true;
        k++;
      }
      if (!luma) continue;
      __syncwarp();
      const int bx0 = (mx * hmax + F->blk_bx[blk]) * 8, by0 = (my * vmax + F->blk_by[blk]) * 8;
      if (!any_ac) {  // DC only: a flat block
        const float v = S.coef[0] * 0.125f + 128.0f;
        const int pv = min(255, max(0, __float2int_rn(v)));
#pragma unroll
        for (int h = 0; h < 2; h++) {
          const int o = lane + 32 * h, px = bx0 + (o & 7), py = by0 + (o >> 3);
          if (px < width && py < height) img[static_cast<size_t>(py) * width + px] = static_cast<uint8_t>(pv);
        }
        continue;
      }
      // A.3.3 inverse DCT, separable: lanes 0..7 take a column each, then a row each (jpeg_idct8, shared with the
      // parallel kernels and the host model)
      if (lane < 8) {
        float in[8], o[8];
#pragma unroll
        for (int v = 0; v < 8; v++) in[v] = S.coef[v * 8 + lane];
        jpeg_idct8(in, o);
#pragma unroll
        for (int y = 0; y < 8; y++) S.tmp[y * 8 + lane] = o[y];
      }
      __syncwarp();
      if (lane < 8) {
        float in[8], o[8];
#pragma unroll
        for (int u = 0; u < 8; u++) in[u] = S.tmp[lane * 8 + u];
        jpeg_idct8(in, o);
        const int py = by0 + lane;
#pragma unroll
        for (int x = 0; x < 8; x++) {
          const int pv = min(255, max(0, __float2int_rn(o[x] + 128.0f)));
          const int px = bx0 + x;
          if (px < width && py < height) img[static_cast<size_t>(py) * width + px] = static_cast<uint8_t>(pv);
        }
      }
    }
    if (++mx == mcus_x) {
      mx = 0;
      my++;
    }
  }
}


// ---- parallel path (streams without restart markers): unstuff -> synchronise -> coefficients -> DC -> IDCT -------------

// exclusive scan over a 1024-thread CTA; returns the prefix of `v`, *total = CTA sum
__device__ __forceinline__ uint32_t cta_exclusive_scan(uint32_t v, uint32_t *warp_sums, uint32_t *total) {
  const int lane = threadIdx.x & 31, wi = threadIdx.x >> 5;
  uint32_t incl = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += t;
  }
  __syncthreads();  // warp_sums may still be read from a previous call
  if (lane == 31) warp_sums[wi] = incl;
  __syncthreads();
  if (wi == 0) {
    uint32_t w = warp_sums[lane];
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t t = __shfl_up_sync(0xffffffffu, w, o);
      if (lane >= o) w += t;
    }
    warp_sums[lane] = w;
  }
  __syncthreads();
  *total = warp_sums[31];
  return incl - v + (wi ? warp_sums[wi - 1] : 0u);
}

// T.81 B.1.1.5: inside the entropy-coded segment FF 00 stands for the byte FF; FF D0..D7 are the RSTn markers between
// restart intervals (E.1.4), which are taken out and remembered as interval starts.  Pass 1 counts the bytes each
// 64-byte chunk keeps (and the markers that end in it), pass 2 turns the counts into offsets, pass 3 moves the bytes.
template <bool SCATTER>
__global__ void __launch_bounds__(256) k_jpeg_unstuff(JpegBatch B) {
  // pass 3 stages the CTA's output (its 256 chunks are consecutive, so is what they keep) in shared memory and writes
  // it out as whole words; +4: the staging area starts at the destination's offset within its first word
  __shared__ __align__(16) uint8_t stage[SCATTER ? 256 * kJpegChunk + 4 : 4];
  const JpegFrame *F = B.frames + blockIdx.y;
  const uint32_t len = F->data_len, nch = (len + kJpegChunk - 1) / kJpegChunk;
  const uint32_t ch0 = blockIdx.x * 256, ch = ch0 + threadIdx.x;
  if (ch0 >= nch) return;
  const bool have = ch < nch;
  const uint8_t *src = B.raw + F->data_off + static_cast<size_t>(ch) * kJpegChunk;
  const uint32_t n = have ? min(kJpegChunk, len - ch * kJpegChunk) : 0u;
  uint32_t prev = (have && ch) ? src[-1] : 0u;
  const uint32_t after = (have && ch * kJpegChunk + n < len) ? src[n] : 0u;  // first byte of the next chunk
  uint4 v[4];
#pragma unroll
  for (int i = 0; i < 4; i++) v[i] = have ? reinterpret_cast<const uint4 *>(src)[i] : make_uint4(0, 0, 0, 0);  // data_off is 16-byte aligned
  const uint32_t *w = reinterpret_cast<const uint32_t *>(v);
  uint8_t *dst = nullptr;
  uint32_t *rst = nullptr;
  uint32_t base = 0, rst_room = 0, cta_base = 0, shift = 0;
  if (SCATTER) {
    cta_base = B.chunk_cnt[F->chunk_off + ch0];
    shift = (F->data_off + cta_base) & 3u;
    if (have) {
      base = B.chunk_cnt[F->chunk_off + ch];
      dst = stage + shift + (base - cta_base);
      const uint32_t r0 = B.chunk_rst[F->chunk_off + ch];
      rst = B.rst_pos + static_cast<size_t>(blockIdx.y) * B.rst_stride + r0;
      rst_room = r0 < B.rst_stride ? B.rst_stride - r0 : 0u;
    }
  }
  uint32_t kept = 0, markers = 0;
#pragma unroll
  for (int i = 0; i < 16; i++) {
#pragma unroll
    for (int j = 0; j < 4; j++) {
      const uint32_t k = 4u * i + j;
      const uint32_t b = (w[i] >> (8 * j)) & 0xffu;
      const uint32_t nb = k + 1 < n ? (j < 3 ? (w[i] >> (8 * ((j + 1) & 3))) & 0xffu : (w[(i + 1) & 15] & 0xffu)) : after;
      const bool in = k < n;
      const bool marker2 = in && prev == 0xffu && b >= 0xd0u && b <= 0xd7u;  // second byte of an RSTn
      const bool marker1 = in && b == 0xffu && nb >= 0xd0u && nb <= 0xd7u;   // first byte of an RSTn
      const bool stuffed = in && b == 0u && prev == 0xffu;
      if (in && !marker1 && !marker2 && !stuffed) {
        if (SCATTER) dst[kept] = static_cast<uint8_t>(b);
        kept++;
      }
      if (marker2) {
        if (SCATTER && markers < rst_room) rst[markers] = base + kept;
        markers++;
      }
      if (in) prev = b;
    }
  }
  if (!SCATTER) {
    if (have) {
      B.chunk_cnt[F->chunk_off + ch] = kept;
      B.chunk_rst[F->chunk_off + ch] = markers;
    }
    return;
  }
  // total kept by the CTA = (offset of the chunk after its last one, or the frame's unstuffed length) - cta_base
  __shared__ uint32_t s_total;
  const uint32_t last = min(nch, ch0 + 256u) - 1u;
  if (ch == last) s_total = base + kept - cta_base;
  __syncthreads();
  const uint32_t total = s_total;
  uint8_t *out = B.clean + F->data_off + cta_base - shift;  // word aligned; stage[i] <-> out[i]
  const uint32_t lo = shift, hi = shift + total;            // valid bytes of the staging area
  const uint32_t w_lo = (lo + 3u) / 4u, w_hi = hi / 4u;     // whole words inside [lo, hi)
  for (uint32_t i = w_lo + threadIdx.x; i < w_hi; i += 256) reinterpret_cast<uint32_t *>(out)[i] = reinterpret_cast<const uint32_t *>(stage)[i];
  if (threadIdx.x < 4) {  // the partial words at both ends, byte by byte
    const uint32_t i = lo + threadIdx.x;
    if (i < min(hi, w_lo * 4u)) out[i] = stage[i];
    const uint32_t t = max(w_hi * 4u, w_lo * 4u) + threadIdx.x;
    if (t < hi && t >= lo) out[t] = stage[t];
  }
}

__global__ void __launch_bounds__(1024) k_jpeg_unstuff_scan(JpegBatch B) {
  __shared__ uint32_t warp_sums[32];
  const JpegFrame *F = B.frames + blockIdx.x;
  const uint32_t nch = (F->data_len + kJpegChunk - 1) / kJpegChunk;
  uint32_t *cnt = B.chunk_cnt + F->chunk_off, *rst = B.chunk_rst + F->chunk_off;
  uint32_t carry = 0, carry_rst = 0;
  for (uint32_t base = 0; base < nch; base += 1024) {
    const uint32_t i = base + threadIdx.x;
    uint32_t total;
    const uint32_t ex = cta_exclusive_scan(i < nch ? cnt[i] : 0u, warp_sums, &total);
    if (i < nch) cnt[i] = carry + ex;
    carry += total;
    const uint32_t exr = cta_exclusive_scan(i < nch ? rst[i] : 0u, warp_sums, &total);
    if (i < nch) rst[i] = carry_rst + exr;
    carry_rst += total;
  }
  if (threadIdx.x == 0) {
    B.clean_len[blockIdx.x] = carry;
    B.nrst[blockIdx.x] = carry_rst;
  }
}

constexpr int kSyncThreads = 128;  // consecutive subsequences per CTA
constexpr int kSyncLocalIters = 48;

// One synchronisation round: every CTA iterates s[i+1] <- f_i(s[i]) on its 128 subsequences to the local fixed point
// (a thread decodes again only when its input state changed), then publishes the states that differ from the stored
// ones.  A round that publishes nothing proves the fixed point.
__global__ void __launch_bounds__(kSyncThreads) k_jpeg_sync(JpegBatch B, int round) {
  __shared__ JpegTables T;
  __shared__ JpegFrame F;
  __shared__ unsigned long long st[kSyncThreads + 1];
  const int f = blockIdx.y, tid = threadIdx.x;
  {
    const uint32_t *src = reinterpret_cast<const uint32_t *>(B.frames + f);
    uint32_t *dst = reinterpret_cast<uint32_t *>(&F);
    for (uint32_t i = tid; i < sizeof(JpegFrame) / 4; i += kSyncThreads) dst[i] = src[i];
  }
  __syncthreads();
  if (F.restart_interval) return;
  uint32_t *changed = B.changed + static_cast<size_t>(f) * kJpegSyncRounds;
  if (round >= 2 && changed[round - 1] == 0) return;  // proven by an earlier round
  const uint32_t end_bits = B.clean_len[f] * 8u;
  const uint32_t nsub = (end_bits + kJpegSubBits - 1) / kJpegSubBits;
  const uint32_t first = blockIdx.x * kSyncThreads;
  if (first + 1 >= nsub) return;
  {
    const uint32_t *src = reinterpret_cast<const uint32_t *>(B.tables + F.tables);
    uint32_t *dst = reinterpret_cast<uint32_t *>(&T);
    for (uint32_t i = tid; i < sizeof(JpegTables) / 4; i += kSyncThreads) dst[i] = src[i];
  }
  const uint32_t i = first + tid;
  const bool active = i + 1 < nsub;  // the last subsequence has no successor
  unsigned long long *sync = B.sync + F.sub_off;
  const uint32_t *words = reinterpret_cast<const uint32_t *>(B.clean + F.data_off);
  auto pack = [](const JpegSyncState &s) { return static_cast<unsigned long long>(s.pos) | (static_cast<unsigned long long>(s.cz) << 32); };
  // states at the start of my subsequence (st[tid]) and of the next CTA's first one (st[128])
  if (i < nsub) st[tid] = (round == 0 || i == 0) ? static_cast<unsigned long long>(i) * kJpegSubBits : sync[i];
  if (tid == kSyncThreads - 1) st[kSyncThreads] = 0xffffffffffffffffull;
  __syncthreads();
  // what this subsequence was last decoded from, and what came out (kept across rounds: a launch whose input did not
  // change has nothing to decode)
  unsigned long long last_in = 0xffffffffffffffffull, out = 0;
  uint32_t nb = 0;
  if (active && round > 0) {
    last_in = B.sync_in[F.sub_off + i];
    out = sync[i + 1];
    nb = B.nblk[F.sub_off + i];
  }
  JpegNullSink none;
  for (int it = 0; it < kSyncLocalIters; it++) {
    const unsigned long long in = active ? st[tid] : 0ull;
    if (active && in != last_in) {
      JpegSyncState s{static_cast<uint32_t>(in), static_cast<uint32_t>(in >> 32)};
      nb = jpeg_decode_span(words, end_bits, (i + 1) * kJpegSubBits, F, T, s, none);
      out = pack(s);
      last_in = in;
    }
    __syncthreads();
    const bool ch = active && st[tid + 1] != out;
    if (ch) st[tid + 1] = out;
    if (!__syncthreads_or(ch)) break;
  }
  if (active) {
    B.nblk[F.sub_off + i] = nb;
    B.sync_in[F.sub_off + i] = last_in;
    // (after kSyncLocalIters without a local fixed point `out` may be stale; the next round continues from it)
    if (round == 0 || sync[i + 1] != out) {
      sync[i + 1] = out;
      changed[round] = 1;
    }
  }
}

// Per frame: is the fixed point proven, and the number of blocks before each subsequence.
__global__ void __launch_bounds__(1024) k_jpeg_blockscan(JpegBatch B) {
  __shared__ uint32_t warp_sums[32];
  const int f = blockIdx.x;
  const JpegFrame *F = B.frames + f;
  bool ok;
  if (F->restart_interval) {  // every interval is decoded from its own start: all that is needed is the right number of markers
    const uint32_t nmcu = static_cast<uint32_t>(F->mcus_x) * F->mcus_y;
    const uint32_t nint = (nmcu + F->restart_interval - 1) / F->restart_interval;
    ok = B.nrst[f] + 1 == nint && B.nrst[f] <= B.rst_stride;
  } else {
    ok = B.changed[static_cast<size_t>(f) * kJpegSyncRounds + kJpegSyncRounds - 1] == 0;
  }
  if (threadIdx.x == 0) B.proven[f] = ok ? 1u : 0u;
  if (!ok || F->restart_interval) return;
  const uint32_t end_bits = B.clean_len[f] * 8u;
  const uint32_t nsub = (end_bits + kJpegSubBits - 1) / kJpegSubBits;
  uint32_t *nblk = B.nblk + F->sub_off;
  uint32_t carry = 0;
  for (uint32_t base = 0; base < nsub; base += 1024) {
    const uint32_t i = base + threadIdx.x;
    const uint32_t v = i + 1 < nsub ? nblk[i] : 0u;
    uint32_t total;
    const uint32_t ex = cta_exclusive_scan(v, warp_sums, &total);
    if (i < nsub) nblk[i] = carry + ex;
    carry += total;
  }
}

// Every subsequence again, this time keeping the luminance coefficients.
__global__ void __launch_bounds__(kSyncThreads) k_jpeg_write(JpegBatch B) {
  __shared__ JpegTables T;
  __shared__ JpegFrame F;
  const int f = blockIdx.y, tid = threadIdx.x;
  if (!B.proven[f]) return;
  {
    const uint32_t *src = reinterpret_cast<const uint32_t *>(B.frames + f);
    uint32_t *dst = reinterpret_cast<uint32_t *>(&F);
    for (uint32_t i = tid; i < sizeof(JpegFrame) / 4; i += kSyncThreads) dst[i] = src[i];
  }
  __syncthreads();
  if (F.restart_interval) return;  // k_jpeg_write_rst
  const uint32_t end_bits = B.clean_len[f] * 8u;
  const uint32_t nsub = (end_bits + kJpegSubBits - 1) / kJpegSubBits;
  if (blockIdx.x * kSyncThreads >= nsub) return;
  {
    const uint32_t *src = reinterpret_cast<const uint32_t *>(B.tables + F.tables);
    uint32_t *dst = reinterpret_cast<uint32_t *>(&T);
    for (uint32_t i = tid; i < sizeof(JpegTables) / 4; i += kSyncThreads) dst[i] = src[i];
  }
  __syncthreads();
  const uint32_t i = blockIdx.x * kSyncThreads + tid;
  if (i >= nsub) return;
  const unsigned long long in = i == 0 ? 0ull : B.sync[F.sub_off + i];
  JpegSyncState s{static_cast<uint32_t>(in), static_cast<uint32_t>(in >> 32)};
  JpegCoefSink sink{B.coef + static_cast<size_t>(f) * B.coef_stride, B.dcs + static_cast<size_t>(f) * (B.coef_stride / 64),
                    B.nblk[F.sub_off + i] / F.nblocks,
                    static_cast<uint32_t>(F.mcus_x) * F.mcus_y, static_cast<uint32_t>(F.hmax) * F.vmax, F.nblocks};
  const uint32_t *words = reinterpret_cast<const uint32_t *>(B.clean + F.data_off);
  jpeg_decode_span(words, end_bits, i + 1 == nsub ? 0xffffffffu : (i + 1) * kJpegSubBits, F, T, s, sink);
}

// Streams with restart markers: an interval starts on a byte boundary with zero predictors (E.1.4), so one thread per
// interval decodes it from its own start -- no synchronisation rounds, absolute DC values written directly.
__global__ void __launch_bounds__(kSyncThreads) k_jpeg_write_rst(JpegBatch B) {
  __shared__ JpegTables T;
  __shared__ JpegFrame F;
  const int f = blockIdx.y, tid = threadIdx.x;
  if (!B.proven[f]) return;
  {
    const uint32_t *src = reinterpret_cast<const uint32_t *>(B.frames + f);
    uint32_t *dst = reinterpret_cast<uint32_t *>(&F);
    for (uint32_t i = tid; i < sizeof(JpegFrame) / 4; i += kSyncThreads) dst[i] = src[i];
  }
  __syncthreads();
  if (!F.restart_interval) return;
  const uint32_t nmcu = static_cast<uint32_t>(F.mcus_x) * F.mcus_y, ri = F.restart_interval;
  const uint32_t nint = (nmcu + ri - 1) / ri;
  if (blockIdx.x * kSyncThreads >= nint) return;
  {
    const uint32_t *src = reinterpret_cast<const uint32_t *>(B.tables + F.tables);
    uint32_t *dst = reinterpret_cast<uint32_t *>(&T);
    for (uint32_t i = tid; i < sizeof(JpegTables) / 4; i += kSyncThreads) dst[i] = src[i];
  }
  __syncthreads();
  const uint32_t k = blockIdx.x * kSyncThreads + tid;
  if (k >= nint) return;
  const uint32_t *rst = B.rst_pos + static_cast<size_t>(f) * B.rst_stride;
  const uint32_t end_bits = B.clean_len[f] * 8u;
  JpegSyncState s{k ? rst[k - 1] * 8u : 0u, 0u};
  const uint32_t limit = k + 1 < nint ? rst[k] * 8u : end_bits;
  JpegIntervalSink sink{{B.coef + static_cast<size_t>(f) * B.coef_stride, B.dcs + static_cast<size_t>(f) * (B.coef_stride / 64), k * ri, nmcu, static_cast<uint32_t>(F.hmax) * F.vmax, F.nblocks}, 0};
  const uint32_t *words = reinterpret_cast<const uint32_t *>(B.clean + F.data_off);
  jpeg_decode_span(words, end_bits, limit, F, T, s, sink, min(ri, nmcu - k * ri) * F.nblocks);
}

// F.2.1.3.1: DC coefficients are coded as differences to the previous block of the component -> running sum over the
// luminance blocks in stream order.
__global__ void __launch_bounds__(1024) k_jpeg_dcscan(JpegBatch B) {
  __shared__ uint32_t warp_sums[32];
  const int f = blockIdx.x;
  if (!B.proven[f]) return;
  const JpegFrame *F = B.frames + f;
  if (F->restart_interval) return;  // k_jpeg_write_rst wrote absolute values
  const uint32_t nlb = static_cast<uint32_t>(F->mcus_x) * F->mcus_y * F->hmax * F->vmax;
  int16_t *dcs = B.dcs + static_cast<size_t>(f) * (B.coef_stride / 64);
  uint32_t carry = 0;
  for (uint32_t base = 0; base < nlb; base += 1024) {
    const uint32_t i = base + threadIdx.x;
    const uint32_t v = i < nlb ? static_cast<uint32_t>(static_cast<int>(dcs[i])) : 0u;  // wraps like int
    uint32_t total;
    const uint32_t ex = cta_exclusive_scan(v, warp_sums, &total);
    if (i < nlb) dcs[i] = static_cast<int16_t>(static_cast<int>(carry + ex + v));
    carry += total;
  }
}

// Dequantisation + A.3.3 inverse DCT + level shift: 8 threads per block (a column each, then a row each), 32 blocks per
// CTA; jpeg_idct8 is shared with the sequential kernel and the host model, so all three give the same bits.  The
// coefficient buffer is handed back all zero.
constexpr int kIdctBlocks = 32;   // blocks per CTA
constexpr int kIdctStride = 72;   // floats per block in shared memory (72 mod 32 = 8: four blocks of a warp on distinct banks)
__global__ void __launch_bounds__(kIdctBlocks * 8) k_jpeg_idct(JpegBatch B) {
  __shared__ __align__(16) float nat[kIdctBlocks * kIdctStride];
  __shared__ __align__(16) float tmp[kIdctBlocks * kIdctStride];
  __shared__ float quant[64];
  __shared__ uint8_t zz[64];
  const int f = blockIdx.y;
  const JpegFrame *F = B.frames + f;
  const int q = threadIdx.x >> 3, j = threadIdx.x & 7, lane = threadIdx.x & 31;
  const uint32_t lb = blockIdx.x * kIdctBlocks + q;
  // every global load of the CTA is issued before the first use of any of them (a CTA lives for a few microseconds:
  // dependent round trips to L2 / HBM would dominate it)
  uint4 *src = reinterpret_cast<uint4 *>(B.coef + static_cast<size_t>(f) * B.coef_stride + static_cast<size_t>(lb) * 64) + j;
  int16_t *dc = B.dcs + static_cast<size_t>(f) * (B.coef_stride / 64) + lb;
  uint4 raw = make_uint4(0, 0, 0, 0);
  uint32_t dcv = 0;
  const bool in_buffer = lb < B.max_luma_blocks;  // inside the frame's slice of the coefficient buffer
  if (in_buffer) {
    raw = *src;
    if (j == 0) dcv = static_cast<uint16_t>(*dc);  // the DC value lives in its own array (and is cleared like the rest)
  }
  const uint32_t proven = B.proven[f];
  const uint32_t hmax = F->hmax, vmax = F->vmax, mcus_x = F->mcus_x, mcus_y = F->mcus_y;
  const int width = F->width, height = F->height;
  float qv = 0.0f;
  if (threadIdx.x < 64) qv = static_cast<float>(F->quant[threadIdx.x]);
  if (!proven) return;
  const uint32_t luma_per_mcu = hmax * vmax;
  const uint32_t nlb = mcus_x * mcus_y * luma_per_mcu;
  if (threadIdx.x < 64) {
    quant[threadIdx.x] = qv;
    zz[threadIdx.x] = c_zigzag[threadIdx.x];
  }
  __syncthreads();
  const bool live = lb < nlb;
  float *mine = nat + q * kIdctStride;
  bool nz_ac = false;
  {
    // coefficients j*8 .. j*8+7 of the block (zigzag order): one 16-byte load, scattered to natural order
    if (live) {
      if (raw.x | raw.y | raw.z | raw.w) *src = make_uint4(0, 0, 0, 0);
      if (j == 0) {
        raw.x = (raw.x & 0xffff0000u) | dcv;
        if (dcv) *dc = 0;
      }
    } else {
      raw = make_uint4(0, 0, 0, 0);
    }
    const uint32_t w[4] = {raw.x, raw.y, raw.z, raw.w};
#pragma unroll
    for (int i = 0; i < 8; i++) {
      const int v = static_cast<int16_t>((w[i >> 1] >> (16 * (i & 1))) & 0xffffu);
      const int k = j * 8 + i, n = zz[k];
      mine[n] = static_cast<float>(v) * quant[n];
      nz_ac = nz_ac || (k > 0 && v != 0);
    }
  }
  const uint32_t acm = __ballot_sync(0xffffffffu, nz_ac);
  const bool ac = ((acm >> (lane & ~7)) & 0xffu) != 0;
  __syncthreads();
  {  // column u = j
    float in[8], o[8];
#pragma unroll
    for (int v = 0; v < 8; v++) in[v] = mine[v * 8 + j];
    jpeg_idct8(in, o);
    float *t = tmp + q * kIdctStride;
#pragma unroll
    for (int y = 0; y < 8; y++) t[y * 8 + j] = o[y];
  }
  __syncthreads();
  if (!live) return;
  // row y = j
  const float4 r0 = *reinterpret_cast<const float4 *>(tmp + q * kIdctStride + j * 8);
  const float4 r1 = *reinterpret_cast<const float4 *>(tmp + q * kIdctStride + j * 8 + 4);
  const float in[8] = {r0.x, r0.y, r0.z, r0.w, r1.x, r1.y, r1.z, r1.w};
  float o[8];
  jpeg_idct8(in, o);
  const float flat = mine[0] * 0.125f + 128.0f;
  uint32_t px8[2] = {0, 0};
#pragma unroll
  for (int x = 0; x < 8; x++) {
    const float val = ac ? o[x] + 128.0f : flat;
    const uint32_t pv = static_cast<uint32_t>(min(255, max(0, __float2int_rn(val))));
    px8[x >> 2] |= pv << (8 * (x & 3));
  }
  const uint32_t mcu = lb / luma_per_mcu, jb = lb % luma_per_mcu;
  const int px = static_cast<int>((mcu % mcus_x) * hmax + F->blk_bx[jb]) * 8;
  const int py = static_cast<int>((mcu / mcus_x) * vmax + F->blk_by[jb]) * 8 + j;
  if (py >= height) return;
  uint8_t *row = B.out + static_cast<size_t>(f) * B.out_stride + static_cast<size_t>(py) * width + px;
  if (px + 8 <= width && (reinterpret_cast<uintptr_t>(row) & 7u) == 0) {
    *reinterpret_cast<uint2 *>(row) = make_uint2(px8[0], px8[1]);
  } else {
    for (int x = 0; x < 8 && px + x < width; x++) row[x] = static_cast<uint8_t>((px8[x >> 2] >> (8 * (x & 3))) & 0xffu);
  }
}

}  // namespace

// Frames whose parallel decode did not reach its fixed point within kJpegSyncRounds rounds (or whose restart markers do
// not add up) are decoded by the sequential warp-per-frame kernel at the end.
void launch_jpeg_decode(const JpegBatch &B, bool any_parallel, cudaStream_t s) {
  if (any_parallel) {
    cudaMemsetAsync(B.changed, 0, sizeof(uint32_t) * kJpegSyncRounds * B.count, s);
    const dim3 gch((B.max_chunks + 255) / 256, B.count);
    k_jpeg_unstuff<false><<<gch, 256, 0, s>>>(B);
    k_jpeg_unstuff_scan<<<B.count, 1024, 0, s>>>(B);
    k_jpeg_unstuff<true><<<gch, 256, 0, s>>>(B);
    const dim3 gsub((B.max_subs + kSyncThreads - 1) / kSyncThreads, B.count);
    for (int r = 0; r < kJpegSyncRounds; r++) k_jpeg_sync<<<gsub, kSyncThreads, 0, s>>>(B, r);
    k_jpeg_blockscan<<<B.count, 1024, 0, s>>>(B);
    k_jpeg_write<<<gsub, kSyncThreads, 0, s>>>(B);
    if (B.max_intervals)
      k_jpeg_write_rst<<<dim3((B.max_intervals + kSyncThreads - 1) / kSyncThreads, B.count), kSyncThreads, 0, s>>>(B);
    k_jpeg_dcscan<<<B.count, 1024, 0, s>>>(B);
    k_jpeg_idct<<<dim3((B.max_luma_blocks + kIdctBlocks - 1) / kIdctBlocks, B.count), kIdctBlocks * 8, 0, s>>>(B);
  }
  k_jpeg_luma<<<B.count, 32, 0, s>>>(B.raw, B.frames, B.tables, B.out, B.out_stride, any_parallel ? B.proven : nullptr);
}

}  // namespace b200tag
