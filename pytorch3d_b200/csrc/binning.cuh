// Exact two-pass tile binning shared by the mesh and point rasterizers.
//
// Role of the reference's coarse stage (pytorch3d/csrc/rasterize_coarse/rasterize_coarse.cu:76-219),
// redesigned: instead of a dense (N, BH, BW, M) table pre-filled with -1 and a brute-force
// element x bin overlap test, every element (face / point) computes the range of pixel centres
// its bounding box can cover (tight to 1e-3 pixel), converts it to a rectangle of 16x16-pixel tiles, and
//   pass 1 (setup+count)  atomically counts elements per tile,
//   pass 2 (scan)         exclusive-scans the counts into segment offsets,
//   pass 3 (fill)         writes element ids into each tile's compact segment,
//   pass 4 (in the fine kernel) the CTA that owns a tile puts its segment in ascending element order.
// No M cap, no overflow drop, no -1 fill; elements whose box contains no pixel centre (most
// sub-pixel triangles) are never binned at all.
#pragma once
#include <climits>

#include "common.cuh"
#include "raster_math.cuh"

namespace b200r {

constexpr uint32_t RECT_EMPTY_X = 0x0000FFFFu;  // tx0 = 0xFFFF > tx1 = 0

// Pixel-index range [lo, hi] that contains every pixel i of an S-pixel axis whose centre pix(i) (as evaluated
// by pix_to_ndc) lies in [vmin, vmax].  The inverse map is evaluated in plain float with a safety margin of
// 1e-3 + 1e-6*S pixels (the float error of either direction is < 2e-4 pixels at S = 512), so the range is a
// superset by at most that margin: binning only has to be conservative, the exact box test happens per
// pixel in the fine pass.  Boxes that contain no pixel centre (most sub-pixel triangles) give lo > hi.
__device__ __forceinline__ void pixel_range(float vmin, float vmax, int S, float range, int& lo, int& hi) {
  const float off = range * 0.5f, scale = (float)S / range, margin = 1e-3f + 1e-6f * (float)S;
  float a = (vmin + off) * scale - 0.5f - margin;
  float b = (vmax + off) * scale - 0.5f + margin;
  a = fminf(fmaxf(a, -1.0f), (float)S + 1.0f);  // also maps NaN to -1 / S+1 (conservative)
  b = fminf(fmaxf(b, -2.0f), (float)S);
  lo = max(0, (int)ceilf(a));
  hi = min(S - 1, (int)floorf(b));
}

// Tile rectangle (in OUTPUT pixel coordinates: xo = W-1-xi, yo = H-1-yi) covering the pixels whose centres
// lie inside [xmin,xmax] x [ymin,ymax] (the reference's per-pixel box test
// `px > xmax || px < xmin || py > ymax || py < ymin`, rasterize_meshes.cu:94-97).
__device__ __forceinline__ uint2 bbox_to_tile_rect(float xmin, float xmax, float ymin, float ymax, int H, int W,
                                                   float rx, float ry) {
  int ix_lo, ix_hi, iy_lo, iy_hi;
  pixel_range(xmin, xmax, W, rx, ix_lo, ix_hi);
  pixel_range(ymin, ymax, H, ry, iy_lo, iy_hi);
  if (ix_lo > ix_hi || iy_lo > iy_hi) return make_uint2(RECT_EMPTY_X, 0u);
  const uint32_t tx0 = (uint32_t)(W - 1 - ix_hi) / TILE, tx1 = (uint32_t)(W - 1 - ix_lo) / TILE;
  const uint32_t ty0 = (uint32_t)(H - 1 - iy_hi) / TILE, ty1 = (uint32_t)(H - 1 - iy_lo) / TILE;
  return make_uint2(tx0 | (tx1 << 16), ty0 | (ty1 << 16));
}

__device__ __forceinline__ bool rect_empty(uint2 r) { return (r.x & 0xFFFFu) > (r.x >> 16); }

// The tile counters are zeroed by a kernel the setup pass is chained to (programmatic dependent launch) instead of a memset
// node: the setup pass's loads and arithmetic overlap it and wait only before their first atomic (binning -1.8 us).
static __global__ void __launch_bounds__(256) zero_ints_kernel(int* __restrict__ p, int64_t n) {
  const int64_t i = ((int64_t)blockIdx.x * 256 + threadIdx.x) * 4;
  pdl_trigger();
  if (i + 4 <= n && (reinterpret_cast<uintptr_t>(p) & 15u) == 0)
    *reinterpret_cast<int4*>(p + i) = make_int4(0, 0, 0, 0);
  else
    for (int64_t j = i; j < n && j < i + 4; ++j) p[j] = 0;
}

// Count one element per tile of its rectangle.  Called by ALL 32 lanes of a warp (lanes without work pass an
// empty rectangle): consecutive elements of a packed mesh are neighbours on screen, so most lanes of a warp
// target the same few tiles -- runs of consecutive lanes that agree are found with a shuffle and a vote (first version:
// all agreeing lanes, with __match_any_sync) and only the first lane of a run issues the atomic, with the run's length.
// This removes the serialisation of thousands of atomics on the hot tiles of a silhouette.
// AGG = false (point clouds, whose packed order carries no spatial coherence): every element simply issues its own
// atomics -- the warp-wide MATCH per round costs more than the 32 uncontended atomics it would merge (8 x 100k
// uniform points: 49 -> see profiles/README.md).
template <bool AGG = true>
__device__ __forceinline__ void warp_count_rect(uint2 r, int n, int TY, int TX, int* __restrict__ tile_count,
                                                int lane) {
  const bool empty = rect_empty(r);
  const int tx0 = r.x & 0xFFFF, tx1 = r.x >> 16, ty0 = r.y & 0xFFFF, ty1 = r.y >> 16;
  if (!AGG) {
    if (empty) return;
    for (int ty = ty0; ty <= ty1; ++ty)
      for (int tx = tx0; tx <= tx1; ++tx) atomicAdd(tile_count + (n * TY + ty) * TX + tx, 1);
    return;
  }
  const int w = empty ? 1 : tx1 - tx0 + 1;
  const int ntile = empty ? 0 : w * (ty1 - ty0 + 1);
  const int rounds = (int)__reduce_max_sync(0xffffffffu, (unsigned)ntile);
  int tx = tx0, ty = ty0;
  for (int i = 0; i < rounds; ++i) {
    const bool act = i < ntile;
    const int t = act ? (n * TY + ty) * TX + tx : -1 - lane;  // inactive lanes get unique keys
    // runs of consecutive lanes with the same tile -- a shuffle and two votes -- instead of __match_any_sync, whose result
    // the atomic waited for (17 % of the setup kernel's stall samples; north-star binning 44.7 -> 40.8 us, config 2 23.6 ->
    // 21.5 us); equal tiles that are not adjacent in the warp cost one more atomic
    const int tprev = __shfl_up_sync(0xffffffffu, t, 1);
    const bool cont = act && lane > 0 && t == tprev;
    const unsigned conts = __ballot_sync(0xffffffffu, cont);
    if (act && !cont) {
      const unsigned after = lane == 31 ? 0u : conts >> (lane + 1);
      atomicAdd(tile_count + t, 1 + (__ffs((int)~after) - 1));
    }
    if (++tx > tx1) {
      tx = tx0;
      ++ty;
    }
  }
}

// Exclusive scan of `counts[0..n)` into `offsets[0..n]` by one CTA of 1024 threads, 8192 elements per sweep
// (eight coalesced loads in flight per thread, then eight block-wide shuffle scans).  `counts` is overwritten
// with the segment starts as well: it becomes the array of fill cursors.
// `order` (optional, n entries): a permutation of the tiles -- long lists first, then short ones, empty tiles last,
// raster order inside each class.  The fine pass runs one CTA per tile and the hardware starts CTAs in index order, so
// its last wave then consists of tiles that finish at once instead of a few heavy ones that leave most SMs idle (a
// blur-band tile of the north-star batch runs for ~120 us of a 920 us kernel).  Keeping the raster order inside a class
// keeps neighbouring tiles -- which share most of their faces' records -- in flight together (an arbitrary order inside
// the classes cost config 5 11 %).  Three classes: longer than the mean non-empty list, shorter, empty; the per-class
// ranks of all tiles come from ONE block scan of a packed counter (3 x 21 bits).
constexpr int ORDER_BITS = 21, ORDER_CLASSES = 3;
__device__ __forceinline__ int order_class(int count, int mean) { return count <= 0 ? 2 : (count > mean ? 0 : 1); }
__device__ __forceinline__ unsigned long long order_key(int count, int mean) {
  return 1ull << (ORDER_BITS * order_class(count, mean));
}

static __global__ void __launch_bounds__(1024) tile_scan_kernel(int* __restrict__ counts, int* __restrict__ offsets, int n,
                                                                int* __restrict__ order) {
  __shared__ long long warp_sums[32];
  __shared__ long long carry_s;
  __shared__ unsigned long long order_sums[32];
  __shared__ unsigned long long order_total, order_carry;
  __shared__ int nonempty_s;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  if (tid == 0) {
    carry_s = 0;
    nonempty_s = 0;
  }
  pdl_trigger();  // (see common.cuh: the fill kernel may become resident now)
  pdl_wait();     // the counters are complete
  __syncthreads();
  // 64-bit running sums, saturated to INT_MAX on output: a batch whose (tile, element) pairs would overflow
  // int32 simply marks the remaining tiles as "does not fit" (they rasterise from the whole mesh range).
  // Every thread owns 8 CONSECUTIVE elements: it scans them in registers, the block scans the 1024 thread
  // totals once (two barriers per sweep of 8192 elements).
  for (int base = 0; base < n; base += 8192) {
    const int i0 = base + tid * 8;
    int v[8];
    // (16-byte accesses: with 4-byte ones every instruction of a warp touched 32 sectors for 128 useful bytes, and the
    // single SM that runs this kernel spent 10 us moving 64 KB)
    const bool vec = i0 + 8 <= n && ((reinterpret_cast<uintptr_t>(counts) | reinterpret_cast<uintptr_t>(offsets)) & 15u) == 0;
    if (vec) {
      const int4 a = *reinterpret_cast<const int4*>(counts + i0), b = *reinterpret_cast<const int4*>(counts + i0 + 4);
      v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w;
      v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
    } else {
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] = i0 + j < n ? counts[i0 + j] : 0;
    }
    long long total = 0;
#pragma unroll
    for (int j = 0; j < 8; ++j) total += v[j];
    if (order != nullptr) {
      int ne = 0;
#pragma unroll
      for (int j = 0; j < 8; ++j) ne += v[j] > 0 ? 1 : 0;
      ne = __reduce_add_sync(0xffffffffu, ne);
      if (lane == 0 && ne > 0) atomicAdd(&nonempty_s, ne);
    }
    long long inc = total;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const long long t = __shfl_up_sync(0xffffffffu, inc, d);
      if (lane >= d) inc += t;
    }
    if (lane == 31) warp_sums[wid] = inc;
    __syncthreads();
    if (wid == 0) {
      long long w = warp_sums[lane];
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        const long long t = __shfl_up_sync(0xffffffffu, w, d);
        if (lane >= d) w += t;
      }
      warp_sums[lane] = w;
    }
    __syncthreads();
    const long long carry = carry_s;
    long long excl = carry + inc - total + (wid > 0 ? warp_sums[wid - 1] : 0);
    int o[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      o[j] = (int)min(excl, (long long)INT_MAX);
      excl += v[j];
    }
    if (vec) {
      const int4 a = make_int4(o[0], o[1], o[2], o[3]), b = make_int4(o[4], o[5], o[6], o[7]);
      *reinterpret_cast<int4*>(offsets + i0) = a;
      *reinterpret_cast<int4*>(offsets + i0 + 4) = b;
      *reinterpret_cast<int4*>(counts + i0) = a;
      *reinterpret_cast<int4*>(counts + i0 + 4) = b;
    } else {
#pragma unroll
      for (int j = 0; j < 8; ++j)
        if (i0 + j < n) {
          offsets[i0 + j] = o[j];
          counts[i0 + j] = o[j];
        }
    }
    __syncthreads();
    if (tid == 0) carry_s = carry + warp_sums[31];
    __syncthreads();
  }
  if (tid == 0) offsets[n] = (int)min(carry_s, (long long)INT_MAX);
  if (order == nullptr) return;
  __syncthreads();  // the offsets written above are visible to the whole CTA; the non-empty count is complete
  const long long total_pairs = carry_s;
  const int mean = (int)min(total_pairs / max(nonempty_s, 1), (long long)INT_MAX);
  // pass 1: how many tiles per class (block reduction of the packed counters)
  unsigned long long mine = 0;
  for (int i = tid; i < n; i += 1024) mine += order_key(offsets[i + 1] - offsets[i], mean);
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) mine += __shfl_xor_sync(0xffffffffu, mine, d);
  if (lane == 0) order_sums[wid] = mine;
  __syncthreads();
  if (tid == 0) {
    unsigned long long t = 0;
    for (int w = 0; w < 32; ++w) t += order_sums[w];
    order_total = t;
    order_carry = 0;
  }
  __syncthreads();
  const unsigned long long total = order_total;
  const unsigned long long fmask = (1ull << ORDER_BITS) - 1;
  long long class_base[ORDER_CLASSES];  // tiles in the classes before this one
  {
    long long at = 0;
#pragma unroll
    for (int c = 0; c < ORDER_CLASSES; ++c) {
      class_base[c] = at;
      at += (long long)((total >> (ORDER_BITS * c)) & fmask);
    }
  }
  // pass 2: ranks inside the classes, in raster order: every thread owns 8 consecutive tiles per sweep
  for (int base = 0; base < n; base += 8192) {
    const int i0 = base + tid * 8;
    unsigned long long k[8], tot = 0;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      k[j] = i0 + j < n ? order_key(offsets[i0 + j + 1] - offsets[i0 + j], mean) : 0ull;
      tot += k[j];
    }
    unsigned long long inc = tot;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const unsigned long long t = __shfl_up_sync(0xffffffffu, inc, d);
      if (lane >= d) inc += t;
    }
    if (lane == 31) order_sums[wid] = inc;
    __syncthreads();
    if (wid == 0) {
      unsigned long long w = order_sums[lane];
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        const unsigned long long t = __shfl_up_sync(0xffffffffu, w, d);
        if (lane >= d) w += t;
      }
      order_sums[lane] = w;
    }
    __syncthreads();
    unsigned long long excl = order_carry + inc - tot + (wid > 0 ? order_sums[wid - 1] : 0ull);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      if (i0 + j < n) {
        long long pos = 0;
#pragma unroll
        for (int c = 0; c < ORDER_CLASSES; ++c)
          if (k[j] == (1ull << (ORDER_BITS * c))) pos = class_base[c] + (long long)((excl >> (ORDER_BITS * c)) & fmask);
        order[pos] = i0 + j;
      }
      excl += k[j];
    }
    __syncthreads();
    if (tid == 0) order_carry += order_sums[31];
    __syncthreads();
  }
}

// Pass 3: scatter element ids into the tile segments (`cursor` starts at each segment's begin).  Same warp
// aggregation as in the count pass: one returning atomic per (warp, tile); the lanes of a group take
// consecutive positions in lane (= element) order.
template <bool AGG>
static __global__ void __launch_bounds__(256)
    tile_fill_kernel(const uint4* __restrict__ rect, int64_t E, int TY, int TX, int* __restrict__ cursor,
                     int* __restrict__ pairs, int64_t capacity) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int lane = threadIdx.x & 31;
  pdl_trigger();  // (see common.cuh: the fine kernel may become resident now)
  pdl_wait();     // the segment starts (scan kernel) and, transitively, the rectangles (setup kernel) are complete
  uint4 r4 = make_uint4(RECT_EMPTY_X, 0u, 0u, 0u);
  if (e < E) r4 = __ldg(rect + e);
  const uint2 r = make_uint2(r4.x, r4.y);
  const bool empty = rect_empty(r);
  const int n = (int)r4.z;
  const int tx0 = r.x & 0xFFFF, tx1 = r.x >> 16, ty0 = r.y & 0xFFFF, ty1 = r.y >> 16;
  if (!AGG) {  // one returning atomic per (element, tile), see warp_count_rect
    if (empty) return;
    for (int ty = ty0; ty <= ty1; ++ty)
      for (int tx = tx0; tx <= tx1; ++tx) {
        const int pos = atomicAdd(cursor + (n * TY + ty) * TX + tx, 1);
        if (pos >= 0 && (int64_t)pos < capacity) pairs[pos] = (int)e;
      }
    return;
  }
  const int w = empty ? 1 : tx1 - tx0 + 1;
  const int ntile = empty ? 0 : w * (ty1 - ty0 + 1);
  const int rounds = (int)__reduce_max_sync(0xffffffffu, (unsigned)ntile);
  int tx = tx0, ty = ty0;
  for (int i = 0; i < rounds; ++i) {
    const bool act = i < ntile;
    const int t = act ? (n * TY + ty) * TX + tx : -1 - lane;
    const int tprev = __shfl_up_sync(0xffffffffu, t, 1);
    const bool cont = act && lane > 0 && t == tprev;
    const unsigned conts = __ballot_sync(0xffffffffu, cont);
    const unsigned heads = __ballot_sync(0xffffffffu, act && !cont);
    // my run's first lane: the highest head at or below me; its length: the continuation bits that follow it
    const int leader = act ? 31 - __clz((int)(heads & (0xffffffffu >> (31 - lane)))) : lane;
    int base = 0;
    if (act && !cont) {
      const unsigned after = lane == 31 ? 0u : conts >> (lane + 1);
      base = atomicAdd(cursor + t, 1 + (__ffs((int)~after) - 1));
    }
    base = __shfl_sync(0xffffffffu, base, leader);
    if (act) {
      const int pos = base + (lane - leader);
      if (pos >= 0 && (int64_t)pos < capacity) pairs[pos] = (int)e;  // (pos < 0: saturated / wrapped cursor)
    }
    if (++tx > tx1) {
      tx = tx0;
      ++ty;
    }
  }
}

// Passes 1 and 3 for elements WITHOUT spatial coherence (point clouds): a CTA takes BIN_CHUNK consecutive elements and
// keeps a private histogram over the tiles of one image in shared memory, so that the thousands of same-address global
// atomics of a dense image (config 3: 1.4 M returning atomics on 8192 counters, 93 % of the fill kernel's stall samples)
// become shared-memory atomics plus one global atomic per touched tile and CTA.  Elements of another image than the
// chunk's first one (a chunk may straddle clouds) use the global counters directly.
// (elements per CTA: config 3 -- 8 x 100 k points -- binning 42.0 us with 2048 = 391 CTAs, 36.7 / 37.4 us with 1024, 37.9 us
// with 512, 48.1 us with 256: more CTAs than SMs x resident CTAs against more global atomics per element)
constexpr int BIN_CHUNK = 1024;        // elements per CTA (4 per thread)
constexpr int BIN_MAX_TILES = 8192;      // tiles per image that the private histogram can hold (32 KB)

// Fill: local histogram -> one returning global atomic per touched tile reserves the CTA's range in the tile's
// segment -> every element takes its place in that range with a shared-memory atomic.
static __global__ void __launch_bounds__(256)
    tile_fill_private_kernel(const uint4* __restrict__ rect, int64_t E, int TY, int TX, int* __restrict__ cursor,
                             int* __restrict__ pairs, int64_t capacity) {
  extern __shared__ int hist[];  // [TY * TX]
  const int tid = threadIdx.x, T = TY * TX;
  const int64_t e0 = (int64_t)blockIdx.x * BIN_CHUNK;
  pdl_trigger();
  for (int t = tid; t < T; t += 256) hist[t] = 0;
  pdl_wait();  // the segment starts (scan kernel) and, transitively, the rectangles (setup kernel) are complete
  __syncthreads();
  const int n0 = (int)__ldg(rect + e0).z;  // the chunk's image (uniform)
  uint2 r[BIN_CHUNK / 256];
  int own[BIN_CHUNK / 256];
#pragma unroll
  for (int i = 0; i < BIN_CHUNK / 256; ++i) {
    const int64_t e = e0 + i * 256 + tid;
    uint4 r4 = make_uint4(RECT_EMPTY_X, 0u, 0u, 0u);
    if (e < E) r4 = __ldg(rect + e);
    r[i] = make_uint2(r4.x, r4.y);
    own[i] = (int)r4.z;
  }
#pragma unroll
  for (int i = 0; i < BIN_CHUNK / 256; ++i) {
    if (rect_empty(r[i]) || own[i] != n0) continue;
    const int tx0 = r[i].x & 0xFFFF, tx1 = r[i].x >> 16, ty0 = r[i].y & 0xFFFF, ty1 = r[i].y >> 16;
    for (int ty = ty0; ty <= ty1; ++ty)
      for (int tx = tx0; tx <= tx1; ++tx) atomicAdd(hist + ty * TX + tx, 1);
  }
  __syncthreads();
  // (four returning atomics in flight per thread: each would wait for its own round trip to L2 otherwise)
  for (int t0 = tid; t0 < T; t0 += 4 * 256) {
    int c[4], b[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) c[u] = t0 + u * 256 < T ? hist[t0 + u * 256] : 0;
#pragma unroll
    for (int u = 0; u < 4; ++u) b[u] = c[u] > 0 ? atomicAdd(cursor + n0 * T + t0 + u * 256, c[u]) : 0;
#pragma unroll
    for (int u = 0; u < 4; ++u)
      if (c[u] > 0) hist[t0 + u * 256] = b[u];  // start of this CTA's range in the tile's segment
  }
  __syncthreads();
#pragma unroll
  for (int i = 0; i < BIN_CHUNK / 256; ++i) {
    if (rect_empty(r[i])) continue;
    const int64_t e = e0 + i * 256 + tid;
    const int tx0 = r[i].x & 0xFFFF, tx1 = r[i].x >> 16, ty0 = r[i].y & 0xFFFF, ty1 = r[i].y >> 16;
    for (int ty = ty0; ty <= ty1; ++ty)
      for (int tx = tx0; tx <= tx1; ++tx) {
        const int pos = own[i] == n0 ? atomicAdd(hist + ty * TX + tx, 1)
                                     : atomicAdd(cursor + (own[i] * TY + ty) * TX + tx, 1);
        if (pos >= 0 && (int64_t)pos < capacity) pairs[pos] = (int)e;  // (pos < 0: saturated / wrapped cursor)
      }
  }
}

// Pass 4 (inside the fine kernels): every tile segment is put in ascending element order by the CTA that
// consumes it.  The fill pass scatters with atomics, so segment order is arbitrary; ascending order makes the fine
// pass visit a pixel's candidates exactly in the order of the reference's naive kernels (rasterize_meshes.cu:301,
// rasterize_points.cu:128), which is what pins tie-breaking and makes the output deterministic.
// "Normalised" bitonic network (every compare-exchange ascending), valid for any segment length:
// partners beyond the end are treated as +inf and skipped.
// (all CTA-wide sorts below are templated on NT, the number of threads of the calling CTA)

// One compare-exchange sweep of the bitonic network over keys[0..n) by the whole CTA.
template <bool MIRROR, int NT>
__device__ __forceinline__ void sort_sweep(int* keys, int n, int d) {
  for (int i = threadIdx.x; i < n; i += NT) {
    const int j = MIRROR ? (i ^ (d - 1)) : (i ^ d);  // MIRROR: d is the block size k
    if (j > i && j < n) {
      const int a = keys[i], b = keys[j];
      if (b < a) {
        keys[i] = b;
        keys[j] = a;
      }
    }
  }
}

// The CTA that owns a tile sorts its list itself -- a separate sort launch cost 19 us of the north-star step.
// Lists of up to 256 faces (one chunk; all but the silhouette tiles) are sorted while they are staged: one key per
// thread, bitonic network ("normalised": every compare-exchange ascending, each merge = a mirror step i ^ (k-1)
// followed by half-cleaners i ^ d), partners closer than 32 by shuffle, the others through shared memory
// (double-buffered: one barrier per step; at most 6 such steps).  Unused threads hold INT_MAX.
template <int NT = TILE_THREADS>
__device__ __forceinline__ int cta_sort256(int key, int n, int* buf) {
  const int i = threadIdx.x;
  int phase = 0;
  for (int k = 2; (k >> 1) < n; k <<= 1) {
    {
      const int m = k - 1;
      int other;
      if (k <= 32) {
        other = __shfl_xor_sync(0xffffffffu, key, m);
      } else {
        buf[phase * NT + i] = key;
        __syncthreads();
        other = buf[phase * NT + (i ^ m)];
        phase ^= 1;
      }
      key = (i & (k >> 1)) == 0 ? min(key, other) : max(key, other);
    }
    for (int d = k >> 2; d > 0; d >>= 1) {
      int other;
      if (d < 32) {
        other = __shfl_xor_sync(0xffffffffu, key, d);
      } else {
        buf[phase * NT + i] = key;
        __syncthreads();
        other = buf[phase * NT + (i ^ d)];
        phase ^= 1;
      }
      key = (i & d) == 0 ? min(key, other) : max(key, other);
    }
  }
  return key;
}

// The same network on 64-bit keys (the point rasterizer sorts a tile's points by (depth, index)): partners closer than
// 32 by two shuffles, the others through shared memory (`buf`: 2 * TILE_THREADS keys).
template <int NT = TILE_THREADS>
__device__ __forceinline__ unsigned long long cta_sort256_u64(unsigned long long key, int n, unsigned long long* buf) {
  const int i = threadIdx.x;
  int phase = 0;
  // keep the smaller key if `low`, the larger otherwise: one 64-bit compare and one select (keys are distinct, or equal
  // padding for which the choice does not matter) instead of a 64-bit min, a max and a select
#define B200R_CE64(other, low) key = (((other) < key) == (low)) ? (other) : key
  for (int k = 2; (k >> 1) < n; k <<= 1) {
    {
      const int m = k - 1;
      unsigned long long other;
      if (k <= 32) {
        other = __shfl_xor_sync(0xffffffffu, key, m);
      } else {
        buf[phase * NT + i] = key;
        __syncthreads();
        other = buf[phase * NT + (i ^ m)];
        phase ^= 1;
      }
      B200R_CE64(other, (i & (k >> 1)) == 0);
    }
    for (int d = k >> 2; d > 0; d >>= 1) {
      unsigned long long other;
      if (d < 32) {
        other = __shfl_xor_sync(0xffffffffu, key, d);
      } else {
        buf[phase * NT + i] = key;
        __syncthreads();
        other = buf[phase * NT + (i ^ d)];
        phase ^= 1;
      }
      B200R_CE64(other, (i & d) == 0);
    }
  }
#undef B200R_CE64
  return key;
}

// Longer lists: the same network swept by the whole CTA over the list in shared memory (when it fits the
// kernel's dynamic shared memory, which is not in use yet) or in place in global memory.
template <int NT = TILE_THREADS>
__device__ __forceinline__ void cta_sort_segment(int* seg, int n, int* s_keys, int cap) {
  const bool in_smem = n <= cap;
  int* keys = in_smem ? s_keys : seg;
  if (in_smem)
    for (int i = threadIdx.x; i < n; i += NT) s_keys[i] = seg[i];
  __syncthreads();
  for (int k = 2; (k >> 1) < n; k <<= 1) {
    sort_sweep<true, NT>(keys, n, k);
    __syncthreads();
    for (int d = k >> 2; d > 0; d >>= 1) {
      sort_sweep<false, NT>(keys, n, d);
      __syncthreads();
    }
  }
  if (in_smem)
    for (int i = threadIdx.x; i < n; i += NT) seg[i] = s_keys[i];
  __syncthreads();
}

// Workspace carving (all int32 / uint2 arrays, 16B-aligned sections).
struct BinWorkspace {
  int* tile_count;  // [ntiles]   counts, then fill cursors (absolute positions)
  int* tile_offset; // [ntiles+1] exclusive offsets; [ntiles] = total pairs
  int* tile_order;  // [ntiles]   tiles by decreasing list length (schedule of the fine pass)
  uint4* rect;      // [E] tile rectangle (x: tx0|tx1<<16, y: ty0|ty1<<16), z: owning mesh / cloud
  int* pairs;       // [capacity]
  int64_t capacity;
  size_t bytes;
};

// Default capacity of the pair buffer: every element in every tile (the exact bound) or, if smaller, 32 pairs per
// element.  (A blur band of 16 pixels puts every sub-pixel face of a 10^6-face mesh into ~9.4 tiles: with the former
// 8 pairs per element the last 12 % of the tiles overflowed and walked the whole mesh -- 64 ms instead of ~10.)
// The buffer is scratch that only the used part of is ever touched.
inline int64_t default_pair_capacity(int64_t E, int N, int H, int W, int tile_h = TILE, int tile_w = TILE) {
  const int64_t tiles = (int64_t)div_up(H, tile_h) * div_up(W, tile_w);
  const int64_t exact = E * tiles;
  const int64_t heur = 32 * E + 64 * (int64_t)N * tiles;
  int64_t c = exact < heur ? exact : heur;
  if (c < 16) c = 16;
  if (c > 0x7fffffff) c = 0x7fffffff;  // positions are int32
  return c;
}

inline BinWorkspace carve_workspace(void* base, int64_t E, int N, int H, int W, int64_t capacity, int tile_h = TILE,
                                    int tile_w = TILE) {
  BinWorkspace ws;
  const int64_t ntiles = (int64_t)N * div_up(H, tile_h) * div_up(W, tile_w);
  if (capacity <= 0) capacity = default_pair_capacity(E, N, H, W, tile_h, tile_w);
  ws.capacity = capacity;
  size_t off = 0;
  char* p = static_cast<char*>(base);
  ws.tile_count = reinterpret_cast<int*>(p + off);
  off = align_up(off + sizeof(int) * (size_t)ntiles, 16);
  ws.tile_offset = reinterpret_cast<int*>(p + off);
  off = align_up(off + sizeof(int) * (size_t)(ntiles + 1), 16);
  ws.tile_order = reinterpret_cast<int*>(p + off);
  off = align_up(off + sizeof(int) * (size_t)ntiles, 16);
  ws.rect = reinterpret_cast<uint4*>(p + off);
  off = align_up(off + sizeof(uint4) * (size_t)(E > 0 ? E : 1), 16);
  ws.pairs = reinterpret_cast<int*>(p + off);
  off = align_up(off + sizeof(int) * (size_t)capacity, 16);
  ws.bytes = off;
  return ws;
}

// Which pixels of a warp's 8x4 footprint lie inside an element's (blur-expanded) box?  One lane tests one face
// against the 8 column and 4 row coordinates of the footprint and builds the 32-bit pixel mask
// (bit = lane of the pixel); the box test is the reference's `px > xmax || px < xmin || ...` (:94-97).
__device__ __forceinline__ unsigned box_pixel_mask(const float4 bx, const float (&col)[8], const float (&row)[4]) {
  unsigned xm = 0, ym = 0;
#pragma unroll
  for (int c = 0; c < 8; ++c) xm |= (!(col[c] > bx.y || col[c] < bx.x) ? 1u : 0u) << c;
#pragma unroll
  for (int r = 0; r < 4; ++r) ym |= (!(row[r] > bx.w || row[r] < bx.z) ? 1u : 0u) << (8 * r);
  return xm * ym;  // ym has one bit per byte, xm < 256: the product replicates xm into the selected rows
}

// Transpose a 32x32 bit matrix held one row per lane (5 butterfly stages of shuffles): afterwards bit k of
// lane l's word is what bit l of lane k's word was.  Turns "pixel mask per face" into "face mask per pixel".
__device__ __forceinline__ unsigned warp_transpose_bits(unsigned a, int lane) {
#pragma unroll
  for (int sft = 16; sft >= 1; sft >>= 1) {
    const unsigned lo = sft == 16 ? 0x0000FFFFu
                      : sft == 8 ? 0x00FF00FFu
                      : sft == 4 ? 0x0F0F0F0Fu
                      : sft == 2 ? 0x33333333u : 0x55555555u;
    const unsigned other = __shfl_xor_sync(0xffffffffu, a, sft);
    a = (lane & sft) ? ((a & ~lo) | ((other & ~lo) >> sft)) : ((a & lo) | ((other & lo) << sft));
  }
  return a;
}

}  // namespace b200r
