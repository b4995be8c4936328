// Blob stage of the B200 AprilTag engine (sm_100a):
//   K7  candidate blobs straight off the blob-pair hash (count limits), segment allocation
//                                                          (reference: apriltag_gpu.cu:522-629,873-905)
//   K8  scatter of the candidates' points into per-blob segments (rank known: no atomics)  (:909-942)
//   K9  one warp / CTA per blob: extents + SelectBlobs (:418-454,534-559), angle keys (:380-412),
//       in-CTA bitonic angle sort, prefix moments, line-fit errors, 7-tap smoothing, peak
//       selection, exhaustive 210-way quad search, corner/area/angle tests
//       (:944-1097, line_fit_filter.cu:22-36,217-278,504-592,709-1193, apriltag_detect.cu:38-282)
// The reference spends 10 CUB device-wide passes and 5 host round trips here; per-blob work is
// independent, so each blob is carried from unsorted points to QuadCorners by a single CTA with
// no host involvement.  Compiled with -fmad=false: the float/double expressions below are
// evaluated exactly as written (IEEE, no contraction), so a CPU restatement reproduces them bit for bit.
#include <cuda_runtime.h>
#include <math_constants.h>
#include <stdint.h>

#include <mutex>

#include "dev_types.h"
#include "kernels.h"

namespace b200tag {

static inline unsigned cdivu(unsigned a, unsigned b) { return (a + b - 1) / b; }
__host__ __device__ constexpr uint32_t next_pow2(uint32_t v) { uint32_t r = 1; while (r < v) r <<= 1; return r; }
constexpr uint32_t kMediumCap = 768;    // medium tier: 128-thread CTA, everything in shared memory
constexpr uint32_t kSortCap = 4096;     // large tier: points sorted / filtered in shared memory

// ---------------------------------------------------------------------------------------------
// K7
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ bool select_blob(const FrameParams &p, uint32_t count, uint32_t minx, uint32_t miny, uint32_t maxx,
                                            uint32_t maxy, int32_t gx, int32_t gy, long long dotsum) {
  // SelectBlobs::operator(), apriltag_gpu.cu:534-559
  if (count < p.min_cluster_pixels) return false;
  if (count > p.max_cluster_pixels) return false;
  if (static_cast<int>((maxx - minx) * (maxy - miny)) < p.min_tag_width) return false;
  // MinMaxExtents::dot(), line_fit_filter.h:51-58
  const long long a = dotsum * 2 - static_cast<long long>(static_cast<int>(minx + maxx) * gx) -
                      static_cast<long long>(static_cast<int>(miny + maxy) * gy);
  const double d = static_cast<double>(a) * 0.5 - 0.05118 * static_cast<double>(gx) + 0.028581 * static_cast<double>(gy);
  const bool quad_reversed = static_cast<float>(d) < 0.0;
  if (!p.reversed_border && quad_reversed) return false;
  if (!p.normal_border && !quad_reversed) return false;
  return true;
}

// One atomic pair per CTA: the per-frame allocation state is packed as
//   alloc = [63:40] clusters | [39:20] candidate blobs | [19:0] small blobs      (large index = blob - small)
// so cluster index, blob index and work-list positions of 256 hash slots come from a single
// 64-bit atomicAdd (the first version issued ~4 returning atomics per warp on one cache line and
// spent 97 % of its time waiting for them).  Only the count limits of SelectBlobs
// (apriltag_gpu.cu:536-541) are applied here; the extent and polarity tests need the blob's
// points and run at the top of the fit kernels.
// (a latency kernel -- two barriers and one round of atomics per trip: eight CTAs per SM and a grid that fills them
//  once, so that every CTA makes as few trips as possible)
__global__ void __launch_bounds__(256, 8) k_select(FrameParams p) {
  __shared__ uint32_t s_warp[8][6];  // per-warp totals: occupied, candidates, small, points, medium, huge
  __shared__ unsigned long long s_base;
  __shared__ uint32_t s_pbase, s_mbase, s_lbase, s_hbase;
  const int frame = blockIdx.y;
  const size_t hoff = static_cast<size_t>(frame) * p.hash_cap;
  Counters *ctr = p.counters + frame;
  b200tag_blob *blobs = p.blobs + static_cast<size_t>(frame) * p.blob_cap;
  WorkItem *small_list = p.small_list + static_cast<size_t>(frame) * p.blob_cap;
  WorkItem *large_list = p.large_list + static_cast<size_t>(frame) * p.blob_cap;
  b200tag_blob *clusters = p.clusters ? p.clusters + static_cast<size_t>(frame) * p.cluster_cap : nullptr;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const uint32_t nocc = min(ctr->num_occupied, p.hash_cap);
  const uint32_t *occupied = p.occupied + hoff;
  // every thread of a CTA runs the same trip count (the loop bound is rounded up to the block size)
  const uint32_t nround = (nocc + blockDim.x - 1) / blockDim.x * blockDim.x;
  for (uint32_t oi = blockIdx.x * blockDim.x + threadIdx.x; oi < nround; oi += gridDim.x * blockDim.x) {
    const bool occ = oi < nocc;
    const uint32_t slot = occ ? occupied[oi] : 0u;
    const unsigned long long key = occ ? p.h_key[hoff + slot] : kEmptyKey;
    b200tag_blob rec;
    bool sel = false;
    if (occ) {
      rec.rep0 = static_cast<uint32_t>(key >> 32);
      rec.rep1 = static_cast<uint32_t>(key);
      rec.min_x = 0xffffffffu; rec.min_y = 0xffffffffu; rec.max_x = 0; rec.max_y = 0;
      rec.count = p.h_count[hoff + slot];
      rec.gx_sum = 0; rec.gy_sum = 0; rec.pxgx_plus_pygy_sum = 0;
      rec.slot = slot;
      rec.offset = 0;
      sel = rec.count >= p.min_cluster_pixels && rec.count <= p.max_cluster_pixels;
      rec.selected = 0;
      // leave the table empty for the next frame
      p.h_key[hoff + slot] = kEmptyKey;
      p.h_count[hoff + slot] = 0;
    }
    const bool small = sel && rec.count <= kSmallBlobPoints;
    const bool medium = sel && !small && rec.count <= kMediumCap;
    const bool huge = sel && rec.count > kSortCap;
    const uint32_t occ_mask = __ballot_sync(0xffffffffu, occ);
    const uint32_t sel_mask = __ballot_sync(0xffffffffu, sel);
    const uint32_t small_mask = __ballot_sync(0xffffffffu, small);
    const uint32_t medium_mask = __ballot_sync(0xffffffffu, medium);
    const uint32_t huge_mask = __ballot_sync(0xffffffffu, huge);
    uint32_t incl = sel ? rec.count : 0u;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += t;
    }
    const uint32_t warp_pts = __shfl_sync(0xffffffffu, incl, 31);
    if (lane == 0) {
      s_warp[warp][0] = __popc(occ_mask);
      s_warp[warp][1] = __popc(sel_mask);
      s_warp[warp][2] = __popc(small_mask);
      s_warp[warp][3] = warp_pts;
      s_warp[warp][4] = __popc(medium_mask);
      s_warp[warp][5] = __popc(huge_mask);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      uint32_t t0 = 0, t1 = 0, t2 = 0, t3 = 0, t4 = 0, t5 = 0;
      for (int w = 0; w < 8; w++) {
        const uint32_t a0 = s_warp[w][0], a1 = s_warp[w][1], a2 = s_warp[w][2], a3 = s_warp[w][3], a4 = s_warp[w][4], a5 = s_warp[w][5];
        s_warp[w][0] = t0; s_warp[w][1] = t1; s_warp[w][2] = t2; s_warp[w][3] = t3; s_warp[w][4] = t4; s_warp[w][5] = t5;  // exclusive prefixes
        t0 += a0; t1 += a1; t2 += a2; t3 += a3; t4 += a4; t5 += a5;
      }
      unsigned long long base = 0;
      uint32_t pb = 0, mb = 0, lb = 0, hb = 0;
      if (t0) {
        const unsigned long long add = (static_cast<unsigned long long>(t0) << 40) | (static_cast<unsigned long long>(t1) << 20) | t2;
        base = atomicAdd(&ctr->alloc, add);
        if (t3) pb = atomicAdd(&ctr->num_seg_points, t3);
        if (t4) mb = atomicAdd(&ctr->num_medium, t4);
        if (t1 - t2 - t4 - t5) lb = atomicAdd(&ctr->num_large, t1 - t2 - t4 - t5);
        if (t5) hb = atomicAdd(&ctr->num_huge, t5);
      }
      s_base = base;
      s_pbase = pb;
      s_mbase = mb;
      s_lbase = lb;
      s_hbase = hb;
    }
    __syncthreads();
    const unsigned long long base = s_base;
    const uint32_t cbase = static_cast<uint32_t>(base >> 40) + s_warp[warp][0];
    const uint32_t bbase = static_cast<uint32_t>(base >> 20) & 0xfffffu;
    const uint32_t sbase = static_cast<uint32_t>(base) & 0xfffffu;
    uint32_t seg_off = 0xffffffffu;
    if (sel) {
      const uint32_t bw = s_warp[warp][1] + __popc(sel_mask & ((1u << lane) - 1u));    // rank among this CTA's blobs
      const uint32_t sw = s_warp[warp][2] + __popc(small_mask & ((1u << lane) - 1u));  // ... among its small blobs
      const uint32_t mw = s_warp[warp][4] + __popc(medium_mask & ((1u << lane) - 1u)); // ... among its medium blobs
      const uint32_t hw = s_warp[warp][5] + __popc(huge_mask & ((1u << lane) - 1u));   // ... among its huge blobs
      // two arrays, four lists: small blobs fill small_list from the front, huge ones from its back;
      // medium blobs fill large_list from the front, large ones from its back
      const uint32_t cta_pos = medium ? s_mbase + mw
                             : (huge ? p.blob_cap - 1u - (s_hbase + hw) : p.blob_cap - 1u - (s_lbase + (bw - sw - mw - hw)));
      const uint32_t b = bbase + bw;
      const uint32_t off = s_pbase + s_warp[warp][3] + incl - rec.count;
      if (b < p.blob_cap && static_cast<uint64_t>(off) + rec.count <= p.point_cap) {
        rec.offset = off;
        blobs[b] = rec;
        seg_off = off;
        const WorkItem item{b, off, rec.count, 0u};
        if (small) small_list[sbase + sw] = item;
        else if (huge) small_list[cta_pos] = item;
        else large_list[cta_pos] = item;
      } else {
        atomicOr(&ctr->status, B200TAG_ST_BLOBS_OVERFLOW);
        // keep the work lists dense: an overflowing blob still occupies its list slot, flagged invalid
        const WorkItem none{0xffffffffu, 0u, 0u, 0u};
        if (small) {
          if (sbase + sw < p.blob_cap) small_list[sbase + sw] = none;
        } else if (cta_pos < p.blob_cap) {
          (huge ? small_list : large_list)[cta_pos] = none;
        }
      }
    }
    if (occ && clusters) {
      const uint32_t c = cbase + __popc(occ_mask & ((1u << lane) - 1u));
      if (c < p.cluster_cap) clusters[c] = rec;
      p.slot_cluster[hoff + slot] = c;
    }
    if (occ) p.slot_off[hoff + slot] = seg_off;
    __syncthreads();  // s_warp / s_base are reused by the next trip
  }
}

// ---------------------------------------------------------------------------------------------
// K8: a candidate blob's points move to its segment; the position is segment start + the rank
// the point was given when it was counted (k_boundary), so there is no atomic and no ordering
// dependence here.  Only the 27 point bits travel on.
// ---------------------------------------------------------------------------------------------
// U points per thread and trip: the chain point -> slot_off[slot] -> store is two dependent memory round trips, and with
// one point per thread the kernel ran at the latency of that chain (0.082 ms per 128 config-2 frames, 53 % of the HBM
// peak); U independent chains per thread hide it.
__global__ void __launch_bounds__(256) k_scatter(FrameParams p) {
  constexpr int U = 4;
  const int frame = blockIdx.y;
  const Counters *ctr = p.counters + frame;
  const uint32_t np = min(ctr->num_points, p.point_cap);
  const uint64_t *points = p.points + static_cast<size_t>(frame) * p.point_cap;
  const uint32_t *slot_off = p.slot_off + static_cast<size_t>(frame) * p.hash_cap;
  uint32_t *seg = p.seg_pts + static_cast<size_t>(frame) * p.point_cap;
  const uint32_t stride = gridDim.x * blockDim.x;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < np; i += U * stride) {
    uint64_t pt[U];
    uint32_t off[U];
#pragma unroll
    for (int u = 0; u < U; u++) {
      const uint32_t j = i + u * stride;
      pt[u] = (j < np && j >= i) ? __ldcs(points + j) : ~0ull;  // all ones: kInvalidSlot
    }
#pragma unroll
    for (int u = 0; u < U; u++) {
      const uint32_t slot = point_slot(pt[u]);
      // slot >= hash_cap: hash overflow (frame already flagged) or past the end
      off[u] = slot < p.hash_cap ? __ldg(slot_off + slot) : 0xffffffffu;
    }
#pragma unroll
    for (int u = 0; u < U; u++)
      if (off[u] != 0xffffffffu) seg[off[u] + point_rank(pt[u])] = point_seg(pt[u]);  // else: NonzeroBlobs, apriltag_gpu.cu:505-518
  }
}

// Debug stages (keep_stages): extents of EVERY blob pair, selected or not, as the reference's C3
// reduce produces them (apriltag_gpu.cu:418-454,829-862), by plain global atomics.
__global__ void __launch_bounds__(256) k_cluster_extents(FrameParams p) {
  const int frame = blockIdx.y;
  const Counters *ctr = p.counters + frame;
  const uint32_t np = min(ctr->num_points, p.point_cap);
  const uint64_t *points = p.points + static_cast<size_t>(frame) * p.point_cap;
  const uint32_t *slot_cluster = p.slot_cluster + static_cast<size_t>(frame) * p.hash_cap;
  b200tag_blob *clusters = p.clusters + static_cast<size_t>(frame) * p.cluster_cap;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < np; i += gridDim.x * blockDim.x) {
    const uint64_t pt = points[i];
    const uint32_t slot = point_slot(pt);
    if (slot >= p.hash_cap) continue;
    const uint32_t c = slot_cluster[slot];
    if (c >= p.cluster_cap) continue;
    const uint32_t sp = point_seg(pt);
    const int x = static_cast<int>(sp_x(sp)), y = static_cast<int>(sp_y(sp));
    const int d = static_cast<int>(sp_dir(sp));
    const int gx = sp_b2w(sp) ? dir_dx(d) : -dir_dx(d), gy = sp_b2w(sp) ? dir_dy(d) : -dir_dy(d);  // points.h:120-125
    b200tag_blob *r = clusters + c;
    atomicMin(&r->min_x, static_cast<uint32_t>(x));
    atomicMax(&r->max_x, static_cast<uint32_t>(x));
    atomicMin(&r->min_y, static_cast<uint32_t>(y));
    atomicMax(&r->max_y, static_cast<uint32_t>(y));
    if (gx) atomicAdd(&r->gx_sum, gx);
    if (gy) atomicAdd(&r->gy_sum, gy);
    const int dot = x * gx + y * gy;
    if (dot) atomicAdd(reinterpret_cast<unsigned long long *>(&r->pxgx_plus_pygy_sum), static_cast<unsigned long long>(static_cast<long long>(dot)));
  }
}

__global__ void __launch_bounds__(256) k_cluster_finish(FrameParams p) {
  const int frame = blockIdx.y;
  const Counters *ctr = p.counters + frame;
  const uint32_t nc = min(alloc_clusters(ctr->alloc), p.cluster_cap);
  b200tag_blob *clusters = p.clusters + static_cast<size_t>(frame) * p.cluster_cap;
  for (uint32_t c = blockIdx.x * blockDim.x + threadIdx.x; c < nc; c += gridDim.x * blockDim.x) {
    b200tag_blob *r = clusters + c;
    r->selected = select_blob(p, r->count, r->min_x, r->min_y, r->max_x, r->max_y, r->gx_sum, r->gy_sum, r->pxgx_plus_pygy_sum);
  }
}

// ---------------------------------------------------------------------------------------------
// K9: blob -> peak table.  Three tiers share one code path (template parameter GS = threads per blob):
//   small  (<= kSmallBlobPoints = 192 points, most blobs): ONE WARP per blob, everything in shared memory,
//          only __syncwarp between phases;
//   medium (<= kMediumCap = 768 points): one 128-thread CTA per blob, everything in shared memory;
//   large  : one 256-thread CTA per blob; sort / errors / peaks in shared memory up to kSortCap = 4096
//          points with the prefix moments in the blob's own (L2-resident) global segment; the rare bigger
//          blob works entirely in its segments of the global arrays.
// Phases: extents + SelectBlobs -> angle keys + bucket sort -> weights + prefix moments -> windowed
// line-fit error -> 7-tap smoothing -> peak list -> [one warp] 10 strongest peaks -> PeakTable for k_quads.
// ---------------------------------------------------------------------------------------------
constexpr int kLargeThreads = 256;
constexpr int kSmallWarps = 4;          // warps (= blobs in flight) per small-tier CTA

template <int GS>
__device__ __forceinline__ void gsync() {
  if constexpr (GS == 32) __syncwarp();
  else __syncthreads();
}

__device__ __forceinline__ void cmpxchg(unsigned long long *a, uint32_t i, uint32_t l) {
  const unsigned long long x = a[i], y = a[l];
  if (x > y) {
    a[i] = y;
    a[l] = x;
  }
}

// All-ascending bitonic network over N = pow2 >= cnt slots; slots >= cnt are virtual +inf and
// never move, so no padding is materialised.  Pair index t always belongs to the same warp
// (t = gt + it * GS) and, for compare distances <= 32, touches only the 64 elements of chunk
// t / 32, so those stages need no block-wide barrier.
template <int GS>
__device__ __noinline__ void bitonic_sort(unsigned long long *a, uint32_t cnt, uint32_t N, uint32_t gt) {
  const uint32_t half = N >> 1;
  for (uint32_t k = 2, lk = 1; k <= N; k <<= 1, lk++) {
    const uint32_t hk = k >> 1;
    for (uint32_t t = gt; t < half; t += GS) {
      const uint32_t blk = t >> (lk - 1), w = t & (hk - 1);
      const uint32_t i = (blk << lk) + w, l = (blk << lk) + k - 1 - w;
      if (l < cnt) cmpxchg(a, i, l);
    }
    // this flip is wide iff k > 64; the following stage (j = k/4, or the next flip if k == 2) is wide iff j >= 64
    if (GS > 32 && (k > 64 || (k == 2 ? false : (k >> 2) >= 64))) __syncthreads();
    else __syncwarp();
    for (uint32_t j = k >> 2; j > 0; j >>= 1) {
      for (uint32_t t = gt; t < half; t += GS) {
        const uint32_t i = ((t & ~(j - 1)) << 1) | (t & (j - 1)), l = i + j;
        if (l < cnt) cmpxchg(a, i, l);
      }
      // next stage: distance j/2, or (after j == 1) the flip of 2k
      const bool this_wide = j >= 64;
      const bool next_wide = (j > 1) ? ((j >> 1) >= 64) : ((k << 1) > 64);
      if (GS > 32 && (this_wide || next_wide)) __syncthreads();
      else __syncwarp();
    }
  }
  gsync<GS>();
}

struct Mom {
  long long Mx, My, W, Mxx, Myy, Mxy;
  int N;
};

// Prefix moments live either in global memory as b200tag_lfp records (large tiers) or, for blobs of at most
// 768 points, in shared memory as six separate arrays: Mxx/Myy/Mxy 64 bit, Mx/My/W 32 bit unsigned
// (W <= 768 * 361 and Mx, My <= W * 8192 < 2^32; the 4096-point low-latency tier is launched only where the same
// bound holds, see launch_blobs), 36 bytes per point instead of 48 and conflict-free.
struct LfStore {
  b200tag_lfp *aos;            // global records, or nullptr
  unsigned long long *m64;     // shared: [3][cap]
  uint32_t *m32;               // shared: [3][cap]
  uint32_t cap;
};
template <bool AOS>
__device__ __forceinline__ b200tag_lfp lf_load(const LfStore &L, uint32_t i) {
  if constexpr (AOS) return L.aos[i];
  b200tag_lfp r;
  r.Mxx = static_cast<long long>(L.m64[i]);
  r.Myy = static_cast<long long>(L.m64[L.cap + i]);
  r.Mxy = static_cast<long long>(L.m64[2 * L.cap + i]);
  r.Mx = L.m32[i];
  r.My = L.m32[L.cap + i];
  r.W = L.m32[2 * L.cap + i];
  return r;
}
template <bool AOS>
__device__ __forceinline__ void lf_store(const LfStore &L, uint32_t i, const b200tag_lfp &r) {
  if constexpr (AOS) {
    L.aos[i] = r;
    return;
  }
  L.m64[i] = static_cast<unsigned long long>(r.Mxx);
  L.m64[L.cap + i] = static_cast<unsigned long long>(r.Myy);
  L.m64[2 * L.cap + i] = static_cast<unsigned long long>(r.Mxy);
  L.m32[i] = static_cast<uint32_t>(r.Mx);
  L.m32[L.cap + i] = static_cast<uint32_t>(r.My);
  L.m32[2 * L.cap + i] = static_cast<uint32_t>(r.W);
}

// ReadMoments, line_fit_filter.cu:745-796 (== CalculateError's window logic, :230-274)
template <bool AOS>
__device__ __forceinline__ Mom read_moments(const LfStore &lf, uint32_t cnt, uint32_t i0, uint32_t i1) {
  Mom m;
  if (i0 < i1) {
    m.N = static_cast<int>(i1 - i0 + 1);
    const b200tag_lfp a = lf_load<AOS>(lf, i1);
    m.Mx = a.Mx; m.My = a.My; m.Mxx = a.Mxx; m.Mxy = a.Mxy; m.Myy = a.Myy; m.W = a.W;
    if (i0 > 0) {
      const b200tag_lfp b = lf_load<AOS>(lf, i0 - 1);
      m.Mx -= b.Mx; m.My -= b.My; m.Mxx -= b.Mxx; m.Mxy -= b.Mxy; m.Myy -= b.Myy; m.W -= b.W;
    }
  } else {
    const b200tag_lfp b = lf_load<AOS>(lf, i0 - 1), z = lf_load<AOS>(lf, cnt - 1), a = lf_load<AOS>(lf, i1);
    m.Mx = z.Mx - b.Mx + a.Mx;
    m.My = z.My - b.My + a.My;
    m.Mxx = z.Mxx - b.Mxx + a.Mxx;
    m.Mxy = z.Mxy - b.Mxy + a.Mxy;
    m.Myy = z.Myy - b.Myy + a.Myy;
    m.W = z.W - b.W + a.W;
    m.N = static_cast<int>(cnt - i0 + i1 + 1);
  }
  return m;
}

// FitLineError (line_fit_filter.cu:22-36) / FitLine (:798-872) / HostFitLine (apriltag_detect.cu:38-90)
__device__ __forceinline__ float eig_small_of(const Mom &m, float *hyp_out, long long *Cxx_o, long long *Cxy_o, long long *Cyy_o) {
  const long long Cxx = m.Mxx * m.W - m.Mx * m.Mx;
  const long long Cxy = m.Mxy * m.W - m.Mx * m.My;
  const long long Cyy = m.Myy * m.W - m.My * m.My;
  const float hyp = hypotf(static_cast<float>(Cxx - Cyy), static_cast<float>(2 * Cxy));
  const float eight_w2 = static_cast<float>(static_cast<double>(m.W * m.W) * 8.0);
  const float eig = (static_cast<float>(Cxx + Cyy) - hyp) / eight_w2;
  if (hyp_out) *hyp_out = hyp;
  if (Cxx_o) { *Cxx_o = Cxx; *Cxy_o = Cxy; *Cyy_o = Cyy; }
  return eig;
}

__device__ __forceinline__ void fit_line(const Mom &m, double *lp01, double *lp23, double *err, double *mse) {
  float hyp;
  long long Cxx, Cxy, Cyy;
  const float eig = eig_small_of(m, &hyp, &Cxx, &Cxy, &Cyy);
  if (lp01) {
    lp01[0] = static_cast<double>(static_cast<float>(m.Mx) / static_cast<float>(m.W * 2));
    lp01[1] = static_cast<double>(static_cast<float>(m.My) / static_cast<float>(m.W * 2));
  }
  if (lp23) {
    const float nx1 = static_cast<float>(Cxx - Cyy) - hyp;
    const float ny1 = static_cast<float>(2 * Cxy);
    const float M1 = nx1 * nx1 + ny1 * ny1;
    const float nx2 = static_cast<float>(2 * Cxy);
    const float ny2 = static_cast<float>(Cyy - Cxx) - hyp;
    const float M2 = nx2 * nx2 + ny2 * ny2;
    float nx, ny;
    if (M1 > M2) { nx = nx1; ny = ny1; } else { nx = nx2; ny = ny2; }
    const float len = hypotf(nx, ny);
    lp23[0] = static_cast<double>(nx / len);
    lp23[1] = static_cast<double>(ny / len);
  }
  *err = static_cast<double>(static_cast<float>(m.N) * eig);
  *mse = static_cast<double>(eig);
}

// TransformLineFitPoint weight, apriltag_gpu.cu:644-657
__device__ __forceinline__ int point_weight(const uint8_t *im, int w, int h, int ix, int iy) {
  int W = 1;
  if (ix > 0 && ix + 1 < w && iy > 0 && iy + 1 < h) {
    const int gx = static_cast<int>(__ldg(im + iy * w + ix + 1)) - static_cast<int>(__ldg(im + iy * w + ix - 1));
    const int gy = static_cast<int>(__ldg(im + (iy + 1) * w + ix)) - static_cast<int>(__ldg(im + (iy - 1) * w + ix));
    // (int)(hypotf(gx, gy) + 1) of the reference.  gx, gy are integers in [-255, 255]: the square root of the exact
    // integer gx^2 + gy^2 is either an integer or at least 1 / (2 * 361) away from one, so the correctly rounded
    // single-precision root gives the same truncation as libdevice's hypotf -- checked for all 511^2 inputs against
    // the oracle's bit-exact hypotf emulation (tests/test_gpu_math.py) -- at a fraction of its instructions.
    W = static_cast<int>(__fsqrt_rn(static_cast<float>(gx * gx + gy * gy)) + 1);
  }
  return W;
}

__device__ __forceinline__ uint32_t float_order(float f) {  // monotone float -> uint map (+0 == -0 after f + 0.0f)
  const uint32_t u = __float_as_uint(f + 0.0f);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

constexpr unsigned long long kNoKey = 0xFFFFFFFFFFFFFFFFull;
constexpr double kDblMax = 1.7976931348623157e308;

// Per-blob scratch of the fit kernels (always in shared memory); WARPS = warps working on the blob.
template <int WARPS>
struct BlobScratch {
  uint32_t peak_idx[kMaxPeaks];
  uint32_t red_u[WARPS > 1 ? WARPS : 1][4];  // per-warp partial extents (CTA tiers only)
  int red_i[WARPS > 1 ? WARPS : 1][3];
  uint32_t npeaks;   // all strict local maxima
  uint32_t nsel;     // min(10, npeaks)
  uint32_t cur;      // work-list position being processed
};

// Scratch of k_quads, one per warp.
struct alignas(16) QuadScratch {
  double seg_err[kMaxPeaks][kMaxPeaks];  // fit error of side (a -> b); kDblMax if mse > max_line_fit_mse
  double seg_nx[kMaxPeaks][kMaxPeaks], seg_ny[kMaxPeaks][kMaxPeaks];
  double lines[4][4];
  float corners[4][2];
  alignas(16) PeakTable t;
};

// nested-loop (Unrank) order of the C(10,4) corner choices, line_fit_filter.cu:709-728
__device__ uint8_t d_combos[kNumCombos][4];

__global__ void k_init_combos() {
  int c = 0;
  for (int m0 = 0; m0 < kMaxPeaks - 3; m0++)
    for (int m1 = m0 + 1; m1 < kMaxPeaks - 2; m1++)
      for (int m2 = m1 + 1; m2 < kMaxPeaks - 1; m2++)
        for (int m3 = m2 + 1; m3 < kMaxPeaks; m3++) {
          d_combos[c][0] = m0; d_combos[c][1] = m1; d_combos[c][2] = m2; d_combos[c][3] = m3;
          c++;
        }
}

constexpr int kPeakRegs = 8;  // peak keys a lane holds in registers during the selection (32 * 8 = 256 peaks)

// The 10 strongest of up to 32 K peaks.  Every lane holds its (up to K) keys of the list in registers, smallest first;
// ten rounds of "warp minimum over the lanes' heads, the owner pops" pick the ten smallest keys -- keys are unique (the
// point index is their low word), so the owner is the lane whose head equals the minimum.  Round r leaves its key in
// lane r: lanes 0..nsel-1 return the chosen peaks, strongest first.
template <int K>
__device__ __forceinline__ unsigned long long top_peaks_regs(const unsigned long long *peaks, uint32_t npk, int lane, uint32_t *nsel_out) {
  static_assert(K == 2 || K == 4 || K == 8, "sorting networks below");
  unsigned long long k[K];
#pragma unroll
  for (int j = 0; j < K; j++) {
    const uint32_t q = static_cast<uint32_t>(lane) + 32u * j;
    k[j] = q < npk ? peaks[q] : kNoKey;
  }
  // optimal sorting networks: 1, 5, 19 comparators
  constexpr int net2[1][2] = {{0, 1}};
  constexpr int net4[5][2] = {{0, 1}, {2, 3}, {0, 2}, {1, 3}, {1, 2}};
  constexpr int net8[19][2] = {{0, 1}, {2, 3}, {4, 5}, {6, 7}, {0, 2}, {1, 3}, {4, 6}, {5, 7}, {1, 2}, {5, 6},
                               {0, 4}, {3, 7}, {1, 5}, {2, 6}, {1, 4}, {3, 6}, {2, 4}, {3, 5}, {3, 4}};
  constexpr int ncmp = K == 2 ? 1 : (K == 4 ? 5 : 19);
#pragma unroll
  for (int c = 0; c < ncmp; c++) {
    const int i0 = K == 2 ? net2[c % 1][0] : (K == 4 ? net4[c % 5][0] : net8[c][0]);
    const int i1 = K == 2 ? net2[c % 1][1] : (K == 4 ? net4[c % 5][1] : net8[c][1]);
    const unsigned long long a = k[i0 % K], b2 = k[i1 % K];
    k[i0 % K] = a < b2 ? a : b2;
    k[i1 % K] = a < b2 ? b2 : a;
  }
  unsigned long long chosen = kNoKey;
  uint32_t nsel = 0;
#pragma unroll 1
  for (int round = 0; round < kMaxPeaks; round++) {
    const uint32_t hi = static_cast<uint32_t>(k[0] >> 32);
    const uint32_t mhi = __reduce_min_sync(0xffffffffu, hi);
    const uint32_t lo = (hi == mhi) ? static_cast<uint32_t>(k[0]) : 0xffffffffu;
    const uint32_t mlo = __reduce_min_sync(0xffffffffu, lo);
    const unsigned long long best = (static_cast<unsigned long long>(mhi) << 32) | mlo;
    if (best == kNoKey) break;
    nsel++;
    if (lane == round) chosen = best;
    if (k[0] == best) {
#pragma unroll
      for (int j = 0; j + 1 < K; j++) k[j] = k[j + 1];
      k[K - 1] = kNoKey;
    }
  }
  *nsel_out = nsel;
  return chosen;
}

// The 10 strongest of MANY (> 256) peaks: ten rounds of a warp-wide minimum over the list; position-ordered
// insertion by lane 0.  Rare (blobs of thousands of points), kept out of line so it does not sit in the hot
// instruction stream.
__device__ __noinline__ uint32_t top_peaks_many(const unsigned long long *peaks, uint32_t npk, uint32_t *peak_idx, int lane) {
  unsigned long long last = 0;
  uint32_t nsel = 0;
#pragma unroll 1
  for (int round = 0; round < kMaxPeaks; round++) {
    unsigned long long best = kNoKey;
#pragma unroll 1
    for (uint32_t i = lane; i < npk; i += 32) {
      const unsigned long long key = peaks[i];
      if ((round == 0 || key > last) && key < best) best = key;
    }
    {  // 64-bit warp minimum as two 32-bit redux steps
      const uint32_t hi = static_cast<uint32_t>(best >> 32);
      const uint32_t mhi = __reduce_min_sync(0xffffffffu, hi);
      const uint32_t lo = (hi == mhi) ? static_cast<uint32_t>(best) : 0xffffffffu;
      const uint32_t mlo = __reduce_min_sync(0xffffffffu, lo);
      best = (static_cast<unsigned long long>(mhi) << 32) | mlo;
    }
    if (best == kNoKey) break;
    last = best;
    nsel++;
    if (lane == 0) {
      const uint32_t v2 = static_cast<uint32_t>(best & 0xffffffffu);
      int q = static_cast<int>(nsel) - 2;
      while (q >= 0 && peak_idx[q] > v2) { peak_idx[q + 1] = peak_idx[q]; q--; }
      peak_idx[q + 1] = v2;
    }
    __syncwarp();
  }
  return nsel;
}

// Working storage of one blob: shared or global memory, chosen by the caller.  Cross-thread hand-offs
// always go through gsync<GS>(), so plain (non-volatile) accesses are sufficient.
struct BlobWork {
  unsigned long long *keys;  // cnt sort keys; dead after the moments phase
  LfStore lf;                // cnt prefix moments
  float *errs;               // cnt weights, then errors
  double *filt;              // cnt filtered errors (may alias keys)
  unsigned long long *peaks; // <= cnt/2 peak keys (may alias errs, which is dead by then)
  bool keys_in_place;        // keys == the blob's segment of p.seg_keys (sorted in place)
  // scratch of the bucket sort; all of it is dead before the prefix moments are written (may alias lf)
  uint32_t *hist;            // hist_cap bucket counters
  uint32_t hist_cap;         // power of two
  uint32_t *tmp;             // 2 * cnt words: theta and in-bucket rank of every point
};

constexpr uint32_t kMaxBucketLoad = 24;  // fuller buckets (thin, elongated blobs) fall back to the bitonic network

// GS = threads per blob; AOS = prefix moments as records in global memory (else shared-memory arrays);
// KEEP = also write the debug stage arrays (keep_stages) -- separate instantiations, so the production
// kernels carry no debug code in their instruction stream.
template <int GS, bool AOS, bool KEEP>
__device__ __forceinline__ void fit_one_blob(const FrameParams &p, int frame, Counters *ctr, uint32_t b, uint32_t cnt, uint32_t off,
                                             b200tag_blob *blob_rec, const BlobWork &wk, BlobScratch<GS / 32> &S, long long *scan, uint32_t gt) {
  const size_t n = static_cast<size_t>(p.w) * p.h;
  const uint8_t *quad = p.quad + frame * n;
  const size_t pbase = static_cast<size_t>(frame) * p.point_cap + off;
  const int lane = threadIdx.x & 31;
  const bool first_warp = gt < 32;

  // (0) the blob's points: extents (MinMaxExtents, apriltag_gpu.cu:418-454) by warp reductions, the
  //     extent / polarity tests of SelectBlobs (:534-559), then the angle keys (:380-412).  The raw
  //     points are parked in the still unused error buffer.
  uint32_t *raw = reinterpret_cast<uint32_t *>(wk.errs);
  {
    // bucket counters of the angle sort (phase 1), zeroed here so that the barrier of the extent reduction covers them too
    const uint32_t N = 1u << (32 - __clz(static_cast<int>(cnt - 1)));  // next power of two (cnt >= 24)
    const uint32_t B = min(N, wk.hist_cap);
    for (uint32_t i = gt; i < B; i += GS) wk.hist[i] = 0;
    if (gt == 0) S.npeaks = 0;
    const uint32_t *sp = p.seg_pts + pbase;
    uint32_t mnx = 0xffffffffu, mxx = 0, mny = 0xffffffffu, mxy = 0;
    int sgx = 0, sgy = 0, sdot = 0;
    for (uint32_t i = gt; i < cnt; i += GS) {
      const uint32_t v = __ldcg(sp + i);
      raw[i] = v;
      const uint32_t x = sp_x(v), y = sp_y(v);
      const int d = static_cast<int>(sp_dir(v));
      const int gx = sp_b2w(v) ? dir_dx(d) : -dir_dx(d), gy = sp_b2w(v) ? dir_dy(d) : -dir_dy(d);  // points.h:120-125
      mnx = min(mnx, x); mxx = max(mxx, x); mny = min(mny, y); mxy = max(mxy, y);
      sgx += gx; sgy += gy;
      sdot += static_cast<int>(x) * gx + static_cast<int>(y) * gy;  // |sum| <= 32768 points * 16382
    }
    mnx = __reduce_min_sync(0xffffffffu, mnx); mxx = __reduce_max_sync(0xffffffffu, mxx);
    mny = __reduce_min_sync(0xffffffffu, mny); mxy = __reduce_max_sync(0xffffffffu, mxy);
    sgx = __reduce_add_sync(0xffffffffu, sgx); sgy = __reduce_add_sync(0xffffffffu, sgy);
    sdot = __reduce_add_sync(0xffffffffu, sdot);
    if constexpr (GS > 32) {
      const int wi = gt >> 5;
      if (lane == 0) {
        S.red_u[wi][0] = mnx; S.red_u[wi][1] = mxx; S.red_u[wi][2] = mny; S.red_u[wi][3] = mxy;
        S.red_i[wi][0] = sgx; S.red_i[wi][1] = sgy; S.red_i[wi][2] = sdot;
      }
      __syncthreads();
      mnx = 0xffffffffu; mxx = 0; mny = 0xffffffffu; mxy = 0; sgx = 0; sgy = 0; sdot = 0;
#pragma unroll
      for (int w = 0; w < GS / 32; w++) {
        mnx = min(mnx, S.red_u[w][0]); mxx = max(mxx, S.red_u[w][1]); mny = min(mny, S.red_u[w][2]); mxy = max(mxy, S.red_u[w][3]);
        sgx += S.red_i[w][0]; sgy += S.red_i[w][1]; sdot += S.red_i[w][2];
      }
    }
    const bool sel = select_blob(p, cnt, mnx, mny, mxx, mxy, sgx, sgy, static_cast<long long>(sdot));
    if (gt == 0) {
      blob_rec->min_x = mnx; blob_rec->min_y = mny; blob_rec->max_x = mxx; blob_rec->max_y = mxy;
      blob_rec->gx_sum = sgx; blob_rec->gy_sum = sgy; blob_rec->pxgx_plus_pygy_sum = sdot;
      blob_rec->selected = sel;
      if (sel) {
        atomicAdd(&ctr->num_selected_blobs, 1u);
        atomicAdd(&ctr->num_selected_points, cnt);
      }
    }
    if (!sel) return;  // uniform across the group
    if constexpr (GS == 32) __syncwarp();  // (CTA tiers: the barrier inside the reduction above)
    // MinMaxExtents::cx/cy, line_fit_filter.h:44-49
    const double cx = static_cast<double>(static_cast<float>(static_cast<int>(mnx + mxx)) * 0.5f) + 0.05118;
    const double cy = static_cast<double>(static_cast<float>(static_cast<int>(mny + mxy)) * 0.5f) + -0.028581;

    // (1) angle sort, C5/C6 (apriltag_gpu.cu:380-412,944-956).  The keys are (theta, dir, y, x); theta is
    //     spread around the whole circle, so a bucket sort does it in O(cnt): B >= cnt buckets over the
    //     theta range (monotone map), in-bucket rank from the counting atomicAdd, exclusive scan, scatter,
    //     then each thread insertion-sorts the few elements of its own buckets on the full 64-bit key.
    // bucket = theta >> bk_shift: theta < 2 * pi * 8e6 + 1 < 2^26, so the B power-of-two buckets cover [0, 2^26) and
    // three quarters of them are in use (average load <= 4/3); a shift instead of a 64-bit multiply and divide
    const uint32_t bk_shift = 26u - (31u - static_cast<uint32_t>(__clz(static_cast<int>(B))));
    uint32_t *th_tmp = wk.tmp, *rk_tmp = wk.tmp + cnt;
#pragma unroll 1
    for (uint32_t i = gt; i < cnt; i += GS) {
      const uint32_t v = raw[i];
      // AddThetaToIndexPoint, apriltag_gpu.cu:400-408
      const float fy = static_cast<float>(static_cast<double>(sp_y(v)) - cy);
      const float fx = static_cast<float>(static_cast<double>(sp_x(v)) - cx);
      const float theta = static_cast<float>((static_cast<double>(atan2f(fy, fx)) + 3.14159265358979323846) * 8e6);
      long long ti = llrintf(theta);
      if (ti < 0) ti = 0;
      const uint32_t th = static_cast<uint32_t>(ti & 0xfffffff);
      const uint32_t bk = (th >> bk_shift);
      th_tmp[i] = th;
      rk_tmp[i] = atomicAdd(&wk.hist[bk], 1u);
    }
    gsync<GS>();
    // exclusive scan of the bucket counts (B / GS consecutive buckets per thread) + fullest bucket
    const uint32_t per = B / GS;  // B and GS are powers of two, B >= GS
    uint32_t sum = 0, mx = 0;
    for (uint32_t j = 0; j < per; j++) {
      const uint32_t c = wk.hist[gt * per + j];
      sum += c;
      mx = max(mx, c);
    }
    uint32_t incl = sum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += t;
    }
    mx = __reduce_max_sync(0xffffffffu, mx);
    if constexpr (GS > 32) {
      const int wi = gt >> 5;
      // (red_u is free: every thread read its phase-0 contents before the barrier that ended the key loop)
      if (lane == 31) S.red_u[wi][0] = incl;
      if (lane == 0) S.red_u[wi][1] = mx;
      __syncthreads();
      uint32_t before = 0;
      mx = 0;
#pragma unroll
      for (int w = 0; w < GS / 32; w++) {
        if (w < wi) before += S.red_u[w][0];
        mx = max(mx, S.red_u[w][1]);
      }
      incl += before;
    }
    const bool bucketed = mx <= kMaxBucketLoad && !(p.test_flags & B200TAG_TEST_BITONIC_SORT);
    if (bucketed) {
      uint32_t ex = incl - sum;
      for (uint32_t j = 0; j < per; j++) {
        const uint32_t c = wk.hist[gt * per + j];
        wk.hist[gt * per + j] = ex;
        ex += c;
      }
      gsync<GS>();
      for (uint32_t i = gt; i < cnt; i += GS) {
        const uint32_t v = raw[i], th = th_tmp[i];
        const uint32_t bk = (th >> bk_shift);
        wk.keys[wk.hist[bk] + rk_tmp[i]] = pack_sort_key(th, sp_dir(v), sp_by(v), sp_bx(v));
      }
      gsync<GS>();
      constexpr uint32_t kRankPer = 6;  // elements a thread can hold in registers across the barrier (192 / 32, 768 / 128)
      if (cnt <= kRankPer * GS) {
        // every element finds its place inside its bucket by counting the smaller keys there (1-2 elements
        // per bucket on average, at most kMaxBucketLoad): balanced across threads, unlike a sort per bucket
        unsigned long long kreg[kRankPer];
        uint32_t preg[kRankPer];
#pragma unroll
        for (uint32_t j = 0; j < kRankPer; j++) {
          const uint32_t q = gt + j * GS;
          kreg[j] = 0;
          preg[j] = 0xffffffffu;
          if (q < cnt) {
            const unsigned long long key = wk.keys[q];
            const uint32_t bk = (key_theta(key) >> bk_shift);
            const uint32_t lo = wk.hist[bk], hi = (bk + 1 < B) ? wk.hist[bk + 1] : cnt;
            uint32_t pos = lo;
#pragma unroll 1
            for (uint32_t i = lo; i < hi; i++) pos += wk.keys[i] < key;
            kreg[j] = key;
            preg[j] = pos;
          }
        }
        gsync<GS>();
#pragma unroll
        for (uint32_t j = 0; j < kRankPer; j++)
          if (preg[j] != 0xffffffffu) wk.keys[preg[j]] = kreg[j];
      } else {
        for (uint32_t j = 0; j < per; j++) {
          const uint32_t bk = gt * per + j;
          const uint32_t lo = wk.hist[bk], hi = (bk + 1 < B) ? wk.hist[bk + 1] : cnt;
          for (uint32_t i = lo + 1; i < hi; i++) {
            const unsigned long long key = wk.keys[i];
            uint32_t q = i;
            while (q > lo && wk.keys[q - 1] > key) {
              wk.keys[q] = wk.keys[q - 1];
              q--;
            }
            wk.keys[q] = key;
          }
        }
      }
      gsync<GS>();
    } else {
      for (uint32_t i = gt; i < cnt; i += GS) {
        const uint32_t v = raw[i];
        wk.keys[i] = pack_sort_key(th_tmp[i], sp_dir(v), sp_by(v), sp_bx(v));
      }
      gsync<GS>();
      bitonic_sort<GS>(wk.keys, cnt, N, gt);
    }
  }
  if (KEEP && !wk.keys_in_place) {
    uint64_t *out = p.seg_keys + pbase;
#pragma unroll 1
    for (uint32_t i = gt; i < cnt; i += GS) out[i] = wk.keys[i];
  }

  // (2) weights and inclusive prefix moments, C7 (apriltag_gpu.cu:631-687,984-987).  Every thread owns a contiguous
  //     chunk of L points (L odd: consecutive threads then hit distinct shared-memory banks): a first pass gathers
  //     the weights and sums the chunk, one scan over the THREADS' totals (a warp scan per warp, the warps' totals
  //     through shared memory) gives each thread its carry-in, a second pass writes the running sums.  Integer sums:
  //     any order gives the reference's values.  (Scanning every 32 points across the warp, as the global-memory
  //     variant below does for the sake of coalesced stores, costs 45 shuffles per 32 points instead of 45 per warp.)
  //     Products: W <= 361, coordinates <= 8192, so W*x fits 32 bits and W*x*x is one 32x32->64 multiply.
  int *wbuf = reinterpret_cast<int *>(wk.errs);
  if constexpr (!AOS) {
    {
      const int wi = static_cast<int>(gt >> 5);
      const uint32_t L = ((cnt + GS - 1) / GS) | 1u;
      const uint32_t c_lo = min(cnt, gt * L), c_hi = min(cnt, c_lo + L);
      unsigned long long t_Mxx = 0, t_Myy = 0, t_Mxy = 0;
      uint32_t t_Mx = 0, t_My = 0, t_W = 0;  // per chunk: L <= 65 points of < 2^22 each
  #pragma unroll 2
      for (uint32_t i = c_lo; i < c_hi; i++) {
        const unsigned long long k = wk.keys[i];
        const uint32_t d = key_dir(k);
        const uint32_t ix2 = 2 * key_bx(k) + dir_dx(d) + 1, iy2 = 2 * key_by(k) + dir_dy(d) + 1;
        const uint32_t W = static_cast<uint32_t>(point_weight(quad, p.w, p.h, static_cast<int>(ix2 / 2), static_cast<int>(iy2 / 2)));
        wbuf[i] = static_cast<int>(W);
        const uint32_t wx = W * ix2, wy = W * iy2;
        t_Mx += wx; t_My += wy; t_W += W;
        t_Mxx += static_cast<unsigned long long>(wx) * ix2;
        t_Mxy += static_cast<unsigned long long>(wx) * iy2;
        t_Myy += static_cast<unsigned long long>(wy) * iy2;
      }
      // inclusive scan of the threads' totals across the warp (64 bit: a blob's Mx, My reach 2^32 above ~1400 points)
      unsigned long long s_Mxx = t_Mxx, s_Myy = t_Myy, s_Mxy = t_Mxy, s_Mx = t_Mx, s_My = t_My, s_W = t_W;
  #pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const unsigned long long u_Mxx = __shfl_up_sync(0xffffffffu, s_Mxx, o), u_Myy = __shfl_up_sync(0xffffffffu, s_Myy, o);
        const unsigned long long u_Mxy = __shfl_up_sync(0xffffffffu, s_Mxy, o);
        // (32-bit shuffles: Mx, My, W of a blob in shared memory stay below 2^32 -- they are stored as 32-bit words)
        const uint32_t u_Mx = __shfl_up_sync(0xffffffffu, static_cast<uint32_t>(s_Mx), o), u_My = __shfl_up_sync(0xffffffffu, static_cast<uint32_t>(s_My), o);
        const uint32_t u_W = __shfl_up_sync(0xffffffffu, static_cast<uint32_t>(s_W), o);
        if (lane >= o) { s_Mx += u_Mx; s_My += u_My; s_W += u_W; s_Mxx += u_Mxx; s_Myy += u_Myy; s_Mxy += u_Mxy; }
      }
      unsigned long long c_Mxx = s_Mxx - t_Mxx, c_Myy = s_Myy - t_Myy, c_Mxy = s_Mxy - t_Mxy;  // carry-in of this thread
      unsigned long long c_Mx = s_Mx - t_Mx, c_My = s_My - t_My, c_W = s_W - t_W;
      if constexpr (GS > 32) {
        unsigned long long *tot = reinterpret_cast<unsigned long long *>(scan);  // [GS / 32][6]
        if (lane == 31) {
          tot[wi * 6 + 0] = s_Mxx; tot[wi * 6 + 1] = s_Myy; tot[wi * 6 + 2] = s_Mxy;
          tot[wi * 6 + 3] = s_Mx;  tot[wi * 6 + 4] = s_My;  tot[wi * 6 + 5] = s_W;
        }
        __syncthreads();
        for (int w = 0; w < wi; w++) {
          c_Mxx += tot[w * 6 + 0]; c_Myy += tot[w * 6 + 1]; c_Mxy += tot[w * 6 + 2];
          c_Mx += tot[w * 6 + 3];  c_My += tot[w * 6 + 4];  c_W += tot[w * 6 + 5];
        }
      }
  #pragma unroll 2
      for (uint32_t i = c_lo; i < c_hi; i++) {
        const unsigned long long k = wk.keys[i];
        const uint32_t d = key_dir(k);
        const uint32_t ix2 = 2 * key_bx(k) + dir_dx(d) + 1, iy2 = 2 * key_by(k) + dir_dy(d) + 1;
        const uint32_t W = static_cast<uint32_t>(wbuf[i]);
        const uint32_t wx = W * ix2, wy = W * iy2;
        c_Mx += wx; c_My += wy; c_W += W;
        c_Mxx += static_cast<unsigned long long>(wx) * ix2;
        c_Mxy += static_cast<unsigned long long>(wx) * iy2;
        c_Myy += static_cast<unsigned long long>(wy) * iy2;
        b200tag_lfp o;
        o.Mxx = static_cast<long long>(c_Mxx); o.Myy = static_cast<long long>(c_Myy); o.Mxy = static_cast<long long>(c_Mxy);
        o.Mx = static_cast<long long>(c_Mx); o.My = static_cast<long long>(c_My); o.W = static_cast<long long>(c_W);
        lf_store<AOS>(wk.lf, i, o);
      }
    }
  } else {
    // Prefix moments in global memory (blobs above the shared-memory capacity): records of 48 bytes, written
    // coalesced -- consecutive lanes own consecutive points.  Weights first (independent strided gathers), then
    // each warp scans its contiguous range 32 points at a time; a first sweep gives the warps' totals.
  #pragma unroll 2
    for (uint32_t i = gt; i < cnt; i += GS) {
      const unsigned long long k = wk.keys[i];
      const uint32_t d = key_dir(k);
      const int ix2 = static_cast<int>(2 * key_bx(k)) + dir_dx(d) + 1, iy2 = static_cast<int>(2 * key_by(k)) + dir_dy(d) + 1;
      wbuf[i] = point_weight(quad, p.w, p.h, ix2 / 2, iy2 / 2);
    }
    gsync<GS>();
    // Inclusive prefix sums by warp scans over 32 consecutive points per step (consecutive lanes touch
    // consecutive shared-memory words: no bank conflicts).  Each warp owns a contiguous range of the blob;
    // in the CTA tiers a first sweep computes the warps' totals, their exclusive scan gives each warp its
    // carry-in.  Products: W <= 361, coordinates <= 8192, so W*x fits 32 bits and W*x*x one 32x32->64 multiply.
    {
      constexpr int kWarps = GS / 32;
      const int wi = static_cast<int>(gt >> 5);
      const uint32_t per_warp = ((cnt + kWarps - 1) / kWarps + 31u) & ~31u;
      const uint32_t w_lo = min(cnt, wi * per_warp), w_hi = min(cnt, w_lo + per_warp);
      unsigned long long c_Mxx = 0, c_Myy = 0, c_Mxy = 0, c_Mx = 0, c_My = 0, c_W = 0;  // carry-in of this warp
      if constexpr (GS > 32) {
        unsigned long long t_Mxx = 0, t_Myy = 0, t_Mxy = 0;
        uint32_t t_Mx = 0, t_My = 0, t_W = 0;  // per lane: at most per_warp / 32 <= 128 points of < 2^22 each
        for (uint32_t i = w_lo + lane; i < w_hi; i += 32) {
          const unsigned long long k = wk.keys[i];
          const uint32_t d = key_dir(k);
          const uint32_t ix2 = 2 * key_bx(k) + dir_dx(d) + 1, iy2 = 2 * key_by(k) + dir_dy(d) + 1;
          const uint32_t W = static_cast<uint32_t>(wbuf[i]);
          const uint32_t wx = W * ix2, wy = W * iy2;
          t_Mx += wx; t_My += wy; t_W += W;
          t_Mxx += static_cast<unsigned long long>(wx) * ix2;
          t_Mxy += static_cast<unsigned long long>(wx) * iy2;
          t_Myy += static_cast<unsigned long long>(wy) * iy2;
        }
        unsigned long long r_Mx = t_Mx, r_My = t_My, r_W = t_W;
  #pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
          t_Mxx += __shfl_xor_sync(0xffffffffu, t_Mxx, o);
          t_Myy += __shfl_xor_sync(0xffffffffu, t_Myy, o);
          t_Mxy += __shfl_xor_sync(0xffffffffu, t_Mxy, o);
          r_Mx += __shfl_xor_sync(0xffffffffu, r_Mx, o);
          r_My += __shfl_xor_sync(0xffffffffu, r_My, o);
          r_W += __shfl_xor_sync(0xffffffffu, r_W, o);
        }
        unsigned long long *tot = reinterpret_cast<unsigned long long *>(scan);  // [kWarps][6]
        if (lane == 0) {
          tot[wi * 6 + 0] = t_Mxx; tot[wi * 6 + 1] = t_Myy; tot[wi * 6 + 2] = t_Mxy;
          tot[wi * 6 + 3] = r_Mx;  tot[wi * 6 + 4] = r_My;  tot[wi * 6 + 5] = r_W;
        }
        __syncthreads();
        for (int w = 0; w < wi; w++) {
          c_Mxx += tot[w * 6 + 0]; c_Myy += tot[w * 6 + 1]; c_Mxy += tot[w * 6 + 2];
          c_Mx += tot[w * 6 + 3];  c_My += tot[w * 6 + 4];  c_W += tot[w * 6 + 5];
        }
      }
  #pragma unroll 1
      for (uint32_t base = w_lo; base < w_hi; base += 32) {
        const uint32_t i = base + lane;
        uint32_t s_Mx = 0, s_My = 0, s_W = 0;
        unsigned long long s_Mxx = 0, s_Myy = 0, s_Mxy = 0;
        if (i < w_hi) {
          const unsigned long long k = wk.keys[i];
          const uint32_t d = key_dir(k);
          const uint32_t ix2 = 2 * key_bx(k) + dir_dx(d) + 1, iy2 = 2 * key_by(k) + dir_dy(d) + 1;
          const uint32_t W = static_cast<uint32_t>(wbuf[i]);
          const uint32_t wx = W * ix2, wy = W * iy2;
          s_Mx = wx; s_My = wy; s_W = W;
          s_Mxx = static_cast<unsigned long long>(wx) * ix2;
          s_Mxy = static_cast<unsigned long long>(wx) * iy2;
          s_Myy = static_cast<unsigned long long>(wy) * iy2;
        }
  #pragma unroll
        for (int o = 1; o < 32; o <<= 1) {  // 32 points of < 2^22 (Mx, My) stay below 2^27: 32-bit scans
          const uint32_t u_Mx = __shfl_up_sync(0xffffffffu, s_Mx, o), u_My = __shfl_up_sync(0xffffffffu, s_My, o);
          const uint32_t u_W = __shfl_up_sync(0xffffffffu, s_W, o);
          const unsigned long long u_Mxx = __shfl_up_sync(0xffffffffu, s_Mxx, o), u_Myy = __shfl_up_sync(0xffffffffu, s_Myy, o);
          const unsigned long long u_Mxy = __shfl_up_sync(0xffffffffu, s_Mxy, o);
          if (lane >= o) { s_Mx += u_Mx; s_My += u_My; s_W += u_W; s_Mxx += u_Mxx; s_Myy += u_Myy; s_Mxy += u_Mxy; }
        }
        if (i < w_hi) {
          b200tag_lfp o;
          o.Mxx = static_cast<long long>(c_Mxx + s_Mxx); o.Myy = static_cast<long long>(c_Myy + s_Myy);
          o.Mxy = static_cast<long long>(c_Mxy + s_Mxy);
          o.Mx = static_cast<long long>(c_Mx + s_Mx); o.My = static_cast<long long>(c_My + s_My); o.W = static_cast<long long>(c_W + s_W);
          lf_store<AOS>(wk.lf, i, o);
        }
        c_Mxx += __shfl_sync(0xffffffffu, s_Mxx, 31); c_Myy += __shfl_sync(0xffffffffu, s_Myy, 31);
        c_Mxy += __shfl_sync(0xffffffffu, s_Mxy, 31);
        c_Mx += __shfl_sync(0xffffffffu, s_Mx, 31); c_My += __shfl_sync(0xffffffffu, s_My, 31); c_W += __shfl_sync(0xffffffffu, s_W, 31);
      }
    }
  }
  gsync<GS>();
  if (KEEP && !AOS) {
    b200tag_lfp *out = p.lfp + pbase;
#pragma unroll 1
    for (uint32_t i = gt; i < cnt; i += GS) out[i] = lf_load<AOS>(wk.lf, i);
  }

  // (3) windowed line-fit error, K10 part 1 (line_fit_filter.cu:217-278)
  const uint32_t ksz = min(20u, cnt / 12u);
#pragma unroll 1
  for (uint32_t i = gt; i < cnt; i += GS) {
    uint32_t i0 = i + cnt - ksz, i1 = i + ksz;  // (i + 2cnt - ksz) % cnt and (i + cnt + ksz) % cnt without division
    if (i0 >= cnt) i0 -= cnt;
    if (i1 >= cnt) i1 -= cnt;
    const Mom m = read_moments<AOS>(wk.lf, cnt, i0, i1);
    const float eig = eig_small_of(m, nullptr, nullptr, nullptr, nullptr);
    wk.errs[i] = static_cast<float>(m.N) * eig;
  }
  gsync<GS>();
  if (KEEP && wk.errs != p.errs + pbase) {
    float *out = p.errs + pbase;
#pragma unroll 1
    for (uint32_t i = gt; i < cnt; i += GS) out[i] = wk.errs[i];
  }
  // (4) 7-tap smoothing in double (:504-525); filt may alias keys, which are dead by now
#pragma unroll 1
  for (uint32_t i = gt; i < cnt; i += GS) {
    const float kf[7] = {0.01110899634659290314f, 0.13533528149127960205f, 0.60653066635131835938f, 1.0f,
                         0.60653066635131835938f, 0.13533528149127960205f, 0.01110899634659290314f};
    double acc = 0.0;
    uint32_t q = i + cnt - 3;  // cnt >= 24 > 3
    if (q >= cnt) q -= cnt;
#pragma unroll
    for (int j = 0; j < 7; j++) {
      const double e = static_cast<double>(wk.errs[q]);
      acc += e * static_cast<double>(kf[j]);
      if (++q == cnt) q = 0;
    }
    wk.filt[i] = acc;
  }
  gsync<GS>();
  if (KEEP && wk.filt != p.filt + pbase) {
    double *out = p.filt + pbase;
#pragma unroll 1
    for (uint32_t i = gt; i < cnt; i += GS) out[i] = wk.filt[i];
  }

  // (5) peak list: strict local maxima (:582), keyed by (-filtered as f32, index) -- C8/C9
  //     (apriltag_gpu.cu:1001-1034).  At most cnt/2 entries.
#pragma unroll 1
  for (uint32_t i = gt; i < cnt; i += GS) {
    const double m = wk.filt[i];
    const double bv = wk.filt[i == 0 ? cnt - 1 : i - 1], av = wk.filt[i + 1 == cnt ? 0 : i + 1];
    if (m > bv && m > av) {
      const uint32_t at = atomicAdd(&S.npeaks, 1u);
      wk.peaks[at] = (static_cast<unsigned long long>(float_order(static_cast<float>(-m))) << 32) | i;
    }
  }
  gsync<GS>();
  const uint32_t npk = S.npeaks;
  if (npk == 0) return;  // no PeakExtents entry -> no FitQuad (uniform across the group)

  // (6) [first warp] the 10 strongest peaks, re-ordered by position, C9/C10 + line_fit_filter.cu:1104-1119.
  //     The slot in the hand-off table is requested now, so the atomic's round trip hides behind the selection.
  uint32_t fq_slot = 0;
  if (first_warp) {
    if (lane == 0) fq_slot = atomicAdd(&ctr->num_fit_quads, 1u);
    uint32_t nsel = 0;
    if (npk <= 32) {
      // one key per lane: bitonic network across the warp, the 10 smallest keys end up in lanes 0..9
      unsigned long long v = lane < static_cast<int>(npk) ? wk.peaks[lane] : kNoKey;
#pragma unroll
      for (int k = 2; k <= 32; k <<= 1) {
#pragma unroll
        for (int j = k >> 1; j > 0; j >>= 1) {
          const unsigned long long other = __shfl_xor_sync(0xffffffffu, v, j);
          const bool take_min = ((lane & k) == 0) == ((lane & j) == 0);
          v = (take_min == (other < v)) ? other : v;
        }
      }
      nsel = min(npk, static_cast<uint32_t>(kMaxPeaks));
      // position order: rank of this lane's point index among the chosen ones
      const uint32_t my_idx = static_cast<uint32_t>(v & 0xffffffffu);
      uint32_t rank = 0;
#pragma unroll
      for (int m = 0; m < kMaxPeaks; m++) {
        const uint32_t o = __shfl_sync(0xffffffffu, my_idx, m);
        rank += (m < static_cast<int>(nsel)) && (o < my_idx);
      }
      if (lane < static_cast<int>(nsel)) S.peak_idx[rank] = my_idx;
    } else if (npk <= 32 * kPeakRegs) {
      // registers per lane sized to the list: 2 (up to 64 peaks), 4 (128) or 8 (256)
      const unsigned long long chosen = npk <= 64    ? top_peaks_regs<2>(wk.peaks, npk, lane, &nsel)
                                        : npk <= 128 ? top_peaks_regs<4>(wk.peaks, npk, lane, &nsel)
                                                     : top_peaks_regs<8>(wk.peaks, npk, lane, &nsel);
      // position order: rank of this lane's point index among the chosen ones
      const uint32_t my_idx = static_cast<uint32_t>(chosen & 0xffffffffu);
      uint32_t rank = 0;
#pragma unroll
      for (int m = 0; m < kMaxPeaks; m++) {
        const uint32_t o = __shfl_sync(0xffffffffu, my_idx, m);
        rank += (m < static_cast<int>(nsel)) && (o < my_idx);
      }
      if (lane < static_cast<int>(nsel)) S.peak_idx[rank] = my_idx;
    } else {
      nsel = top_peaks_many(wk.peaks, npk, S.peak_idx, lane);
    }
    if (lane == 0) S.nsel = nsel;
    __syncwarp();
  }

  // hand-off to k_quads: the chosen peaks and the prefix-moment records around them
  if (first_warp) {
    const uint32_t nm = S.nsel;
    const uint32_t fq = __shfl_sync(0xffffffffu, fq_slot, 0);
    if (fq < p.blob_cap) {
      PeakTable *t = p.peak_tables + static_cast<size_t>(frame) * p.blob_cap + fq;
      if (lane == 0) {
        t->blob = b; t->cnt = cnt; t->nsel = nm; t->npk = npk; t->rep0 = blob_rec->rep0; t->rep1 = blob_rec->rep1;
        t->last = lf_load<AOS>(wk.lf, cnt - 1);
      }
      if (lane < static_cast<int>(nm)) {
        const uint32_t i = S.peak_idx[lane];
        t->idx[lane] = i;
        t->at[lane] = lf_load<AOS>(wk.lf, i);
        b200tag_lfp z;
        z.Mxx = 0; z.Myy = 0; z.Mxy = 0; z.Mx = 0; z.My = 0; z.W = 0;
        t->before[lane] = i > 0 ? lf_load<AOS>(wk.lf, i - 1) : z;
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------
// K10: quad search.  One warp per blob that has peaks, fed by the fit kernels' PeakTable: the work
// per blob no longer depends on its size (<= 90 side fits, 210 corner choices, 4 corners), so it
// runs as a separate, uniformly loaded kernel instead of as a serial tail of every fit CTA.
// ---------------------------------------------------------------------------------------------
// ReadMoments (line_fit_filter.cu:745-796) for the range from chosen peak a to chosen peak c.
__device__ __forceinline__ Mom table_moments(const PeakTable &T, int a, int c) {
  const uint32_t i0 = T.idx[a], i1 = T.idx[c];
  const b200tag_lfp hi = T.at[c], lo = T.before[a];
  Mom m;
  if (i0 < i1) {
    m.N = static_cast<int>(i1 - i0 + 1);
    m.Mx = hi.Mx; m.My = hi.My; m.Mxx = hi.Mxx; m.Mxy = hi.Mxy; m.Myy = hi.Myy; m.W = hi.W;
    if (i0 > 0) { m.Mx -= lo.Mx; m.My -= lo.My; m.Mxx -= lo.Mxx; m.Mxy -= lo.Mxy; m.Myy -= lo.Myy; m.W -= lo.W; }
  } else {
    const b200tag_lfp z = T.last;
    m.Mx = z.Mx - lo.Mx + hi.Mx;
    m.My = z.My - lo.My + hi.My;
    m.Mxx = z.Mxx - lo.Mxx + hi.Mxx;
    m.Mxy = z.Mxy - lo.Mxy + hi.Mxy;
    m.Myy = z.Myy - lo.Myy + hi.Myy;
    m.W = z.W - lo.W + hi.W;
    m.N = static_cast<int>(T.cnt - i0 + i1 + 1);
  }
  return m;
}

constexpr int kQuadWarps = 4;

__global__ void __launch_bounds__(kQuadWarps * 32, 8) k_quads(FrameParams p) {
  __shared__ QuadScratch s_q[kQuadWarps];
  const int frame = blockIdx.y;
  const int lane = threadIdx.x & 31;
  QuadScratch &S = s_q[threadIdx.x >> 5];
  Counters *ctr = p.counters + frame;
  const uint32_t nfq = min(ctr->num_fit_quads, p.blob_cap);
  const PeakTable *tables = p.peak_tables + static_cast<size_t>(frame) * p.blob_cap;
  for (uint32_t fq = blockIdx.x * kQuadWarps + (threadIdx.x >> 5); fq < nfq; fq += gridDim.x * kQuadWarps) {
    __syncwarp();
    {  // the table into shared memory: every lane issues all of its 16-byte loads before the first store
      constexpr uint32_t kPieces = sizeof(PeakTable) / 16, kPer = (kPieces + 31) / 32;
      const uint4 *src = reinterpret_cast<const uint4 *>(tables + fq);
      uint4 *dst = reinterpret_cast<uint4 *>(&S.t);
      uint4 v[kPer];
#pragma unroll
      for (uint32_t k = 0; k < kPer; k++)
        if (lane + 32 * k < kPieces) v[k] = __ldcg(src + lane + 32 * k);
#pragma unroll
      for (uint32_t k = 0; k < kPer; k++)
        if (lane + 32 * k < kPieces) dst[lane + 32 * k] = v[k];
    }
    __syncwarp();
    const PeakTable &T = S.t;
    const uint32_t b = T.blob, cnt = T.cnt, npk = T.npk;

  // (7) side-fit table: every ordered pair of chosen peaks (<= 90 fits instead of 4 per combination), enumerated
  //     densely (pair t = (a, c'), c' skipping a) so that nm (nm - 1) fits take ceil(nm (nm - 1) / 32) rounds.  Only
  //     forward pairs (a < c) can be a first or second side, whose normals the corner test needs; the others are
  //     closing sides (peak m3 back to m0): error only.
  const int nm = static_cast<int>(T.nsel);
  const double max_mse = static_cast<double>(p.max_line_fit_mse);
  const uint32_t inv_nm1 = nm > 1 ? 65535u / static_cast<uint32_t>(nm - 1) + 1u : 0u;  // t / (nm - 1) for t < 90, exactly
  for (int t = lane; t < nm * (nm - 1); t += 32) {
    const int a = static_cast<int>((static_cast<uint32_t>(t) * inv_nm1) >> 16);
    int c = t - a * (nm - 1);
    c += c >= a;
    const Mom mo = table_moments(T, a, c);
    double err, mse, nrm[2] = {0.0, 0.0};
    fit_line(mo, nullptr, a < c ? nrm : nullptr, &err, &mse);
    S.seg_err[a][c] = (mse > max_mse) ? kDblMax : err;  // line_fit_filter.cu:964-966,1009,1027,1035
    S.seg_nx[a][c] = nrm[0];
    S.seg_ny[a][c] = nrm[1];
  }
  __syncwarp();

  // (8) [first warp] exhaustive search over the C(10,4) corner choices, K11 (line_fit_filter.cu:976-1048,1161)
  {
    const double max_dot = static_cast<double>(p.cos_critical_rad);
    double my_err = kDblMax;
    int my_rank = kNumCombos;
    for (int c = lane; c < kNumCombos; c += 32) {
      const uchar4 cm = *reinterpret_cast<const uchar4 *>(d_combos[c]);
      const int m0 = cm.x, m1 = cm.y, m2 = cm.z, m3 = cm.w;
      if (m3 >= nm) continue;
      const double e01 = S.seg_err[m0][m1];
      if (e01 == kDblMax) continue;
      const double e12 = S.seg_err[m1][m2];
      if (e12 == kDblMax) continue;
      const double dot = S.seg_nx[m0][m1] * S.seg_nx[m1][m2] + S.seg_ny[m0][m1] * S.seg_ny[m1][m2];
      if (fabs(dot) > max_dot) continue;
      const double e23 = S.seg_err[m2][m3];
      if (e23 == kDblMax) continue;
      const double e30 = S.seg_err[m3][m0];
      if (e30 == kDblMax) continue;
      const double tot = e01 + e12 + e23 + e30;
      if (tot < my_err) { my_err = tot; my_rank = c; }  // ranks ascend per lane: ties keep the lowest
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const double oe = __shfl_xor_sync(0xffffffffu, my_err, o);
      const int orank = __shfl_xor_sync(0xffffffffu, my_rank, o);
      if (oe < my_err || (oe == my_err && orank < my_rank)) { my_err = oe; my_rank = orank; }
    }

    // (9) FitQuad, then UpdateFitQuads + AdjustPixelCenters (apriltag_detect.cu:98-282): lanes 0..3 fit
    //     one side each and intersect one corner each; lane 0 runs the quad tests.
    const double best = my_err;
    const int bi = my_rank < kNumCombos ? my_rank : 0;
    const bool valid = best < static_cast<double>(p.max_line_fit_mse * static_cast<float>(cnt));
    b200tag_fit_quad *fqo = (fq < p.blob_cap) ? (p.fit_quads + static_cast<size_t>(frame) * p.blob_cap + fq) : nullptr;
    if (lane == 0 && fqo) {
      fqo->blob_index = b;
      fqo->valid = valid;
      fqo->num_peaks = static_cast<int32_t>(npk);
      fqo->err = best;
    }
    if (lane < 4) {
      uint32_t i0 = 0;
      Mom mo;
      if (valid) {
        i0 = T.idx[d_combos[bi][lane]];
        mo = table_moments(T, d_combos[bi][lane], d_combos[bi][(lane + 1) & 3]);  // line_fit_filter.cu:1188-1191
        double err, mse;
        fit_line(mo, S.lines[lane], S.lines[lane] + 2, &err, &mse);
      }
      if (fqo) {
        fqo->indices[lane] = i0;
        b200tag_moments mm = b200tag_moments{0, 0, 0, 0, 0, 0, 0, 0};
        if (valid) { mm.Mx = mo.Mx; mm.My = mo.My; mm.W = mo.W; mm.Mxx = mo.Mxx; mm.Myy = mo.Myy; mm.Mxy = mo.Mxy; mm.N = mo.N; }
        fqo->moments[lane] = mm;
      }
    }
    __syncwarp();
    if (valid) {
      bool bad = false;
      if (lane < 4) {  // apriltag_detect.cu:125-166
        const int i = lane, nx = (lane + 1) & 3;
        const double A00 = S.lines[i][3], A01 = -S.lines[nx][3];
        const double A10 = -S.lines[i][2], A11 = S.lines[nx][2];
        const double B0 = -S.lines[i][0] + S.lines[nx][0];
        const double B1 = -S.lines[i][1] + S.lines[nx][1];
        const double det = A00 * A11 - A10 * A01;
        const double W00 = A11 / det, W01 = -A01 / det;
        if (fabs(det) < 0.001) bad = true;
        const double L0 = W00 * B0 + W01 * B1;
        S.corners[i][0] = static_cast<float>(S.lines[i][0] + L0 * A00);
        S.corners[i][1] = static_cast<float>(S.lines[i][1] + L0 * A10);
      }
      bad = __any_sync(0xffffffffu, bad);
      __syncwarp();
      // the six edge lengths of the two triangles of the area test, one lane each (hypotf is the expensive part of the
      // tests below): (0,1) (1,2) (2,0) | (2,3) (3,0) (0,2)
      float elen = 0;
      if (lane < 6) {
        const int a = (0x032210 >> (4 * lane)) & 0xf, c = (0x203021 >> (4 * lane)) & 0xf;
        elen = hypotf(S.corners[c][0] - S.corners[a][0], S.corners[c][1] - S.corners[a][1]);
      }
      float elens[6];
#pragma unroll
      for (int i = 0; i < 6; i++) elens[i] = __shfl_sync(0xffffffffu, elen, i);
      if (lane == 0 && !bad) {
        float cr[4][2];
        for (int j = 0; j < 4; j++) { cr[j][0] = S.corners[j][0]; cr[j][1] = S.corners[j][1]; }
        {  // :171-207
          float area = 0;
          float pp;
          pp = (elens[0] + elens[1] + elens[2]) / 2;
          area += sqrtf(pp * (pp - elens[0]) * (pp - elens[1]) * (pp - elens[2]));
          pp = (elens[3] + elens[4] + elens[5]) / 2;
          area += sqrtf(pp * (pp - elens[3]) * (pp - elens[4]) * (pp - elens[5]));
          if (static_cast<double>(area) < 0.95 * p.min_tag_width * p.min_tag_width) bad = true;
        }
        if (!bad) {  // :209-238
          for (int i = 0; i < 4; i++) {
            const int i0 = i, i1 = (i + 1) & 3, i2 = (i + 2) & 3;
            const float dx1 = cr[i1][0] - cr[i0][0], dy1 = cr[i1][1] - cr[i0][1];
            const float dx2 = cr[i2][0] - cr[i1][0], dy2 = cr[i2][1] - cr[i1][1];
            const float cos_dtheta = (dx1 * dx2 + dy1 * dy2) / sqrtf((dx1 * dx1 + dy1 * dy1) * (dx2 * dx2 + dy2 * dy2));
            if (fabsf(cos_dtheta) > p.cos_critical_rad || dx1 * dy2 < dy1 * dx2) { bad = true; break; }
          }
        }
        if (!bad) {
          const float f = static_cast<float>(p.f);
          if (f > 1) {  // AdjustPixelCenters, :260-282
            for (int j = 0; j < 4; j++) {
              cr[j][0] = (cr[j][0] - 0.5f) * f + 0.5f;
              cr[j][1] = (cr[j][1] - 0.5f) * f + 0.5f;
            }
          }
          const uint32_t qi = atomicAdd(&ctr->num_quads, 1u);
          if (qi < p.quad_cap) {
            b200tag_quad &q = (p.quads + static_cast<size_t>(frame) * p.quad_cap)[qi];
            for (int j = 0; j < 4; j++) { q.corners[j][0] = cr[j][0]; q.corners[j][1] = cr[j][1]; }
            q.reversed_border = p.reversed_border && !p.normal_border;
            q.blob_index = b;
            q.rep0 = T.rep0;
            q.rep1 = T.rep1;
          } else {
            atomicOr(&ctr->status, B200TAG_ST_QUADS_OVERFLOW);
          }
        }
      }
    }
  }
  }
}

// ---- small tier: one warp per blob ------------------------------------------------------------
struct SmallWarpShared {
  unsigned long long keys[kSmallBlobPoints];  // sort keys, later the filtered errors (same size)
  unsigned long long lf64[3 * kSmallBlobPoints];  // prefix moments (LfStore); bucket-sort scratch before that
  uint32_t lf32[3 * kSmallBlobPoints];
  alignas(16) float errs[kSmallBlobPoints];   // weights -> errors -> peak list (8-byte keys)
  BlobScratch<1> scratch;
};

template <bool KEEP>
__global__ void __launch_bounds__(kSmallWarps * 32, 6) k_fit_small(FrameParams p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  SmallWarpShared &S = reinterpret_cast<SmallWarpShared *>(smem_raw)[threadIdx.x >> 5];
  const int frame = blockIdx.y;
  const int lane = threadIdx.x & 31;
  Counters *ctr = p.counters + frame;
  b200tag_blob *blobs = p.blobs + static_cast<size_t>(frame) * p.blob_cap;
  const WorkItem *list = p.small_list + static_cast<size_t>(frame) * p.blob_cap;
  const uint32_t nlist = min(alloc_small(ctr->alloc), p.blob_cap);
  BlobWork wk;
  wk.keys = S.keys;
  wk.lf.aos = nullptr; wk.lf.m64 = S.lf64; wk.lf.m32 = S.lf32; wk.lf.cap = kSmallBlobPoints;
  wk.errs = S.errs;
  wk.filt = reinterpret_cast<double *>(S.keys);
  wk.peaks = reinterpret_cast<unsigned long long *>(S.errs);
  wk.keys_in_place = false;
  wk.hist = reinterpret_cast<uint32_t *>(S.lf64);
  wk.hist_cap = next_pow2(kSmallBlobPoints);
  wk.tmp = wk.hist + next_pow2(kSmallBlobPoints);
  uint32_t nxt = 0;
  if (lane == 0) nxt = atomicAdd(&ctr->next_small, 1u);
  while (true) {
    __syncwarp();
    const uint32_t li = __shfl_sync(0xffffffffu, nxt, 0);
    if (li >= nlist) break;
    if (lane == 0) nxt = atomicAdd(&ctr->next_small, 1u);  // the next item's round trip overlaps this blob
    const WorkItem item = list[li];
    const uint32_t b = item.blob, off = item.offset, cnt = item.count;
    if (b >= p.blob_cap) continue;  // overflow marker
    // On a blob-list overflow (frame flagged B200TAG_ST_BLOBS_OVERFLOW) the huge tier's entries, which fill this
    // list from its back, can reach into the range read here; this tier's buffers hold kSmallBlobPoints points.
    if (cnt > kSmallBlobPoints) continue;
    fit_one_blob<32, false, KEEP>(p, frame, ctr, b, cnt, off, blobs + b, wk, S.scratch, nullptr, lane);
  }
}

// ---- CTA tiers: one CTA per blob ----------------------------------------------------------------
//   medium: 128 threads, blobs of 193..768 points, everything in shared memory (5 CTAs per SM)
//   large : 256 threads, blobs above 768 points; sort / errors / peaks in shared memory up to 4096 points,
//           prefix moments in the blob's own L2-resident segment (3 CTAs per SM)
// k_select sorts the blobs into the tiers' work lists (medium from the front of large_list, large from its back).
// Shared memory of a CTA tier: one buffer, carved per blob in one of two ways --
//   layout A (blobs of at most LF_CAP points, everything in shared memory):
//       keys[LF_CAP] u64 | prefix moments 3 x u64[LF_CAP], 3 x u32[LF_CAP] | errs[LF_CAP] f32     (48 bytes per point)
//   layout B (blobs of at most KEY_CAP > LF_CAP points, prefix moments in the blob's global segment):
//       keys[KEY_CAP] u64 | errs[KEY_CAP] f32 | bucket counters / warp totals of the scans
// so that a tier whose size range spans both (large: A up to 1536 points, B up to 4096) pays for the larger of the two,
// not their sum.
template <int THREADS, uint32_t KEY_CAP, uint32_t LF_CAP>
struct CtaShared {
  static constexpr bool kHasB = KEY_CAP > LF_CAP;
  // layout B scratch (64-bit words): KEY_CAP bucket counters of the angle sort if that beats the warp totals' 6 * THREADS
  static constexpr uint32_t kScanWords = kHasB ? (KEY_CAP / 2 > 6 * THREADS ? KEY_CAP / 2 : 6 * THREADS) : 0;
  static constexpr size_t kBytesA = static_cast<size_t>(LF_CAP) * 48;
  static constexpr size_t kBytesB = kHasB ? static_cast<size_t>(KEY_CAP) * 12 + static_cast<size_t>(kScanWords) * 8 : 0;
  alignas(16) unsigned char buf[kBytesA > kBytesB ? kBytesA : kBytesB];
  long long tot[6 * (THREADS / 32)];  // layout A: warp totals of the prefix scan
  BlobScratch<THREADS / 32> scratch;

  __device__ unsigned long long *a_keys() { return reinterpret_cast<unsigned long long *>(buf); }
  __device__ unsigned long long *a_lf64() { return reinterpret_cast<unsigned long long *>(buf) + LF_CAP; }
  __device__ uint32_t *a_lf32() { return reinterpret_cast<uint32_t *>(buf + static_cast<size_t>(LF_CAP) * 32); }
  __device__ float *a_errs() { return reinterpret_cast<float *>(buf + static_cast<size_t>(LF_CAP) * 44); }
  __device__ unsigned long long *b_keys() { return reinterpret_cast<unsigned long long *>(buf); }
  __device__ float *b_errs() { return reinterpret_cast<float *>(buf + static_cast<size_t>(KEY_CAP) * 8); }
  __device__ long long *b_scan() { return reinterpret_cast<long long *>(buf + static_cast<size_t>(KEY_CAP) * 12); }
};
static_assert(kMediumCap % 4 == 0 && kSortCap % 4 == 0, "16-byte alignment of the carved arrays");

template <int THREADS, uint32_t KEY_CAP, uint32_t LF_CAP, uint32_t MIN_CNT, uint32_t MAX_CNT, int MIN_CTAS, bool KEEP>
__global__ void __launch_bounds__(THREADS, MIN_CTAS) k_fit_cta(FrameParams p, int tier) {
  using Shared = CtaShared<THREADS, KEY_CAP, LF_CAP>;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  Shared &S = *reinterpret_cast<Shared *>(smem_raw);
  const int frame = blockIdx.y;
  const int tid = threadIdx.x;
  Counters *ctr = p.counters + frame;
  b200tag_blob *blobs = p.blobs + static_cast<size_t>(frame) * p.blob_cap;
  // tier 0: medium (front of large_list), 1: large (back of large_list), 2: huge (back of small_list)
  const WorkItem *list = (tier == 2 ? p.small_list : p.large_list) + static_cast<size_t>(frame) * p.blob_cap;
  const uint32_t nlist = min(tier == 0 ? ctr->num_medium : (tier == 1 ? ctr->num_large : ctr->num_huge), p.blob_cap);
  // bucket counters of blobs whose prefix moments live in global memory: the scan scratch, largest power of two
  constexpr uint32_t kScanHist = (KEY_CAP / 2 > 6 * THREADS) ? KEY_CAP : ((6u * THREADS * 2u >= 2048u) ? 2048u : 1024u);
  uint32_t *next = tier == 0 ? &ctr->next_medium : (tier == 1 ? &ctr->next_large : &ctr->next_huge);
  uint32_t nxt = 0;
  if (tid == 0) nxt = atomicAdd(next, 1u);
  while (true) {
    __syncthreads();
    if (tid == 0) S.scratch.cur = nxt;
    __syncthreads();
    const uint32_t li = S.scratch.cur;
    if (li >= nlist) break;
    if (tid == 0) nxt = atomicAdd(next, 1u);  // the next item's round trip overlaps this blob
    const WorkItem item = list[tier == 0 ? li : p.blob_cap - 1u - li];
    const uint32_t b = item.blob, blob_off = item.offset, blob_cnt = item.count;
    if (b >= p.blob_cap) continue;  // overflow marker
    if (blob_cnt < MIN_CNT || blob_cnt > MAX_CNT) continue;  // (cannot happen: k_select sorts blobs into tiers)
    const size_t pbase = static_cast<size_t>(frame) * p.point_cap + blob_off;
    BlobWork wk;
    // branches that the tier's size limits rule out are not compiled (each one is a full copy of the fit code)
    constexpr bool kHasSmemLf = LF_CAP > 0;
    constexpr bool kHasGlobalLf = MAX_CNT > LF_CAP;
    constexpr bool kHasInPlace = MAX_CNT > KEY_CAP;
    // layout A keeps Mx, My, W as 32-bit words: cnt points of weight <= 361 and coordinate <= 2 max(w, h) + 1 must stay
    // below 2^32 (always true up to 1452 points; tiers without a fallback are launched only where it holds)
    const bool lf32_ok = LF_CAP <= 1452 || !kHasGlobalLf ||
                         static_cast<uint64_t>(blob_cnt) * 361u * (2u * static_cast<uint32_t>(max(p.w, p.h)) + 1u) < (1ull << 32);
    if (kHasSmemLf && blob_cnt <= LF_CAP && lf32_ok) {  // everything in shared memory
      wk.keys = S.a_keys(); wk.errs = S.a_errs();
      wk.lf.aos = nullptr; wk.lf.m64 = S.a_lf64(); wk.lf.m32 = S.a_lf32(); wk.lf.cap = LF_CAP;
      wk.filt = reinterpret_cast<double *>(S.a_keys());
      wk.peaks = reinterpret_cast<unsigned long long *>(S.a_errs());
      wk.keys_in_place = false;
      wk.hist = reinterpret_cast<uint32_t *>(S.a_lf64()); wk.hist_cap = next_pow2(LF_CAP > 0 ? LF_CAP : 1); wk.tmp = wk.hist + next_pow2(LF_CAP > 0 ? LF_CAP : 1);
      fit_one_blob<THREADS, false, KEEP>(p, frame, ctr, b, blob_cnt, blob_off, blobs + b, wk, S.scratch, S.tot, tid);
    } else if (kHasGlobalLf && KEY_CAP > LF_CAP && blob_cnt <= KEY_CAP) {  // prefix moments in the blob's global segment
      wk.keys = S.b_keys(); wk.errs = S.b_errs();
      wk.lf.aos = p.lfp + pbase; wk.lf.m64 = nullptr; wk.lf.m32 = nullptr; wk.lf.cap = 0;
      wk.filt = reinterpret_cast<double *>(S.b_keys());
      wk.peaks = reinterpret_cast<unsigned long long *>(S.b_errs());
      wk.keys_in_place = false;
      wk.hist = reinterpret_cast<uint32_t *>(S.b_scan()); wk.hist_cap = kScanHist; wk.tmp = reinterpret_cast<uint32_t *>(p.lfp + pbase);
      fit_one_blob<THREADS, true, KEEP>(p, frame, ctr, b, blob_cnt, blob_off, blobs + b, wk, S.scratch, S.b_scan(), tid);
    } else if (kHasInPlace) {  // too large for shared memory: work in place in the global arrays
      wk.keys = reinterpret_cast<unsigned long long *>(p.seg_keys + pbase);
      wk.lf.aos = p.lfp + pbase; wk.lf.m64 = nullptr; wk.lf.m32 = nullptr; wk.lf.cap = 0;
      wk.errs = p.errs + pbase; wk.filt = p.filt + pbase;
      wk.peaks = reinterpret_cast<unsigned long long *>(p.peak_ws + static_cast<size_t>(frame) * (p.point_cap / 2 + 1) + blob_off / 2);
      wk.keys_in_place = true;
      wk.hist = reinterpret_cast<uint32_t *>(S.b_scan()); wk.hist_cap = kScanHist; wk.tmp = reinterpret_cast<uint32_t *>(p.lfp + pbase);
      fit_one_blob<THREADS, true, KEEP>(p, frame, ctr, b, blob_cnt, blob_off, blobs + b, wk, S.scratch, S.b_scan(), tid);
    }
  }
}

using MediumShared = CtaShared<128, kMediumCap, kMediumCap>;
constexpr uint32_t kLargeLfCap = 1536;  // large tier: blobs up to here entirely in shared memory (72 KB = the 4096-point layout B + 8 KB)
using LargeShared = CtaShared<kLargeThreads, kSortCap, kLargeLfCap>;
static_assert(sizeof(LargeShared) <= 76800 - 1024, "three CTAs of the large tier per SM");
// six CTAs of either tier per SM: 228 KB less 1 KB per CTA
static_assert(sizeof(MediumShared) <= 37888, "shared memory of the medium tier");
#define K_FIT_MEDIUM(KEEP) k_fit_cta<128, kMediumCap, kMediumCap, kSmallBlobPoints + 1, kMediumCap, 6, KEEP>
#define K_FIT_LARGE(KEEP) k_fit_cta<kLargeThreads, kSortCap, kLargeLfCap, kMediumCap + 1, kSortCap, 3, KEEP>
// (measured: blobs up to 2304 points entirely in shared memory at TWO CTAs per SM, 0.436 -> 0.522 ms per 128 frames)
// huge: 512 threads, blobs above 4096 points (clutter, image-spanning edges); keys / errors / peaks in shared memory up
// to 8192 points (one CTA per SM), beyond that in place in the global arrays
constexpr int kHugeThreads = 512;
constexpr uint32_t kHugeCap = 8192;
using HugeShared = CtaShared<kHugeThreads, kHugeCap, 0>;
// (held to 64 registers -- this instance has the global-memory path only and fits without spills -- so that a resident
//  huge-tier CTA leaves half the register file to the other tiers' CTAs; a 256-thread variant was slower: 0.46 -> 0.67 ms
//  per 16 config-5 frames)
#define K_FIT_HUGE(KEEP) k_fit_cta<kHugeThreads, kHugeCap, 0, kSortCap + 1, 0xffffffffu, (KEEP) ? 1 : 2, KEEP>
// large tier for one or a few frames at a time (the node's case: one Detect per camera frame): the same blobs on 512
// threads.  A frame has a few dozen of them, far fewer than SMs, so the time of the blob stage is the time of ONE blob;
// twice the threads nearly halve it (single frame: 111 -> 6x us), while in batches, where CTAs outnumber SMs many times,
// the 256-thread kernel above is the better one.
// With one CTA per SM there is room for the prefix moments in shared memory too (36 B x 4096 points = 147 KB of 216 KB).
using Large512Shared = CtaShared<kHugeThreads, kSortCap, kSortCap>;
#define K_FIT_LARGE512(KEEP) k_fit_cta<kHugeThreads, kSortCap, kSortCap, kMediumCap + 1, kSortCap, 1, KEEP>
static_assert(sizeof(Large512Shared) <= 227 * 1024, "shared memory of the low-latency large tier");
constexpr int kLowLatencyFrames = 4;  // batches up to this size take the 512-thread large tier

void launch_blobs_init(cudaStream_t s) {
  static bool dev_ready[64] = {false};
  static std::mutex mu;  // detectors may be created from several threads
  std::lock_guard<std::mutex> lock(mu);
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev >= 0 && dev < 64 && !dev_ready[dev]) {
    cudaFuncSetAttribute(k_fit_small<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(sizeof(SmallWarpShared) * kSmallWarps));
    cudaFuncSetAttribute(k_fit_small<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(sizeof(SmallWarpShared) * kSmallWarps));
    cudaFuncSetAttribute(K_FIT_MEDIUM(false), cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(sizeof(MediumShared)));
    cudaFuncSetAttribute(K_FIT_MEDIUM(true), cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(sizeof(MediumShared)));
    cudaFuncSetAttribute(K_FIT_LARGE(false), cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(sizeof(LargeShared)));
    cudaFuncSetAttribute(K_FIT_LARGE(true), cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(sizeof(LargeShared)));
    cudaFuncSetAttribute(K_FIT_HUGE(false), cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(sizeof(HugeShared)));
    cudaFuncSetAttribute(K_FIT_HUGE(true), cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(sizeof(HugeShared)));
    cudaFuncSetAttribute(K_FIT_LARGE512(false), cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(sizeof(Large512Shared)));
    cudaFuncSetAttribute(K_FIT_LARGE512(true), cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(sizeof(Large512Shared)));
    k_init_combos<<<1, 1, 0, s>>>();
    dev_ready[dev] = true;
  }
}

void launch_blobs(const FrameParams &p, int frames, Launcher &ln, const SideStreams *side) {
  const cudaStream_t s = ln.s;
  ln.timed("select", [&] { k_select<<<dim3(max(1u, min(16u, 148u * 8u / static_cast<unsigned>(frames))), frames), 256, 0, s>>>(p); });
  ln.timed("scatter", [&] { k_scatter<<<dim3(max(8u, min(592u, cdivu(4736u, frames))), frames), 256, 0, s>>>(p); });
  if (p.clusters) {  // debug stage only (keep_stages)
    ln.untimed([&] { k_cluster_extents<<<dim3(max(8u, min(592u, cdivu(4736u, frames))), frames), 256, 0, s>>>(p); });
    ln.untimed([&] { k_cluster_finish<<<dim3(16, frames), 256, 0, s>>>(p); });
  }
  // The three tiers are independent and each is latency bound at modest occupancy: with side streams they run
  // concurrently (largest blobs first), so their tails overlap; the per-kernel timing mode runs them serially.
  // Resident capacity per SM: 5 small-tier CTAs (4 warps = 4 blobs each), 5 medium-tier CTAs, 3 large-tier CTAs.
  const bool fork = side && side->s[0] && side->s[1] && side->s[2];
  cudaStream_t s_large = fork ? side->s[0] : s, s_medium = fork ? side->s[1] : s, s_huge = fork ? side->s[2] : s;
  if (fork) {
    cudaEventRecord(side->fork, s);
    cudaStreamWaitEvent(s_large, side->fork, 0);
    cudaStreamWaitEvent(s_medium, side->fork, 0);
    cudaStreamWaitEvent(s_huge, side->fork, 0);
  }
  ln.timed("fit_huge", [&] {
    const dim3 g(max(1u, min(148u, cdivu(592u, frames))), frames);
    if (p.keep_stages) K_FIT_HUGE(true)<<<g, kHugeThreads, sizeof(HugeShared), s_huge>>>(p, 2);
    else K_FIT_HUGE(false)<<<g, kHugeThreads, sizeof(HugeShared), s_huge>>>(p, 2);
  });
  // (the shared-memory prefix moments keep Mx, My, W as 32-bit words: kSortCap points of weight <= 361 must not reach
  //  2^32, which holds for quad images up to 1451 pixels a side -- larger frames take the 256-thread kernel)
  const bool lf32_ok = static_cast<uint64_t>(kSortCap) * 361u * (2u * static_cast<uint32_t>(max(p.w, p.h)) + 1u) < (1ull << 32);
  ln.timed("fit_large", [&] {
    if (frames <= kLowLatencyFrames && lf32_ok) {
      const dim3 g(max(1u, min(148u, cdivu(592u, frames))), frames);
      if (p.keep_stages) K_FIT_LARGE512(true)<<<g, kHugeThreads, sizeof(Large512Shared), s_large>>>(p, 1);
      else K_FIT_LARGE512(false)<<<g, kHugeThreads, sizeof(Large512Shared), s_large>>>(p, 1);
    } else {
      const dim3 g(max(3u, min(444u, cdivu(1776u, frames))), frames);
      if (p.keep_stages) K_FIT_LARGE(true)<<<g, kLargeThreads, sizeof(LargeShared), s_large>>>(p, 1);
      else K_FIT_LARGE(false)<<<g, kLargeThreads, sizeof(LargeShared), s_large>>>(p, 1);
    }
  });
  const dim3 g(max(4u, min(740u, cdivu(2960u, frames))), frames);
  ln.timed("fit_medium", [&] {
    if (p.keep_stages) K_FIT_MEDIUM(true)<<<g, 128, sizeof(MediumShared), s_medium>>>(p, 0);
    else K_FIT_MEDIUM(false)<<<g, 128, sizeof(MediumShared), s_medium>>>(p, 0);
  });
  ln.timed("fit_small", [&] {
    if (p.keep_stages) k_fit_small<true><<<g, kSmallWarps * 32, sizeof(SmallWarpShared) * kSmallWarps, s>>>(p);
    else k_fit_small<false><<<g, kSmallWarps * 32, sizeof(SmallWarpShared) * kSmallWarps, s>>>(p);
  });
  if (fork) {
    cudaEventRecord(side->join[0], s_large);
    cudaEventRecord(side->join[1], s_medium);
    cudaEventRecord(side->join[2], s_huge);
    cudaStreamWaitEvent(s, side->join[0], 0);
    cudaStreamWaitEvent(s, side->join[1], 0);
    cudaStreamWaitEvent(s, side->join[2], 0);
  }
  ln.timed("quads", [&] { k_quads<<<dim3(max(2u, min(592u, cdivu(2368u, frames))), frames), kQuadWarps * 32, 0, s>>>(p); });
}

}  // namespace b200tag
