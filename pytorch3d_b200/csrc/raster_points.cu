// Point-cloud rasterizer for sm_100a: setup/bin pass, per-tile fine pass (top-K per pixel), backward.
//
// Replaces, behind the same operator signature, the reference's
//   PointBoundingBoxKernel + RasterizeCoarseCudaKernel   (rasterize_coarse.cu:53-74, 76-219)
//   RasterizePointsFineCudaKernel / NaiveCudaKernel       (rasterize_points.cu:223-298, 87-149)
//   RasterizePointsBackwardCudaKernel                     (rasterize_points.cu:366-411)
// Same skeleton as raster_meshes.cu: exact tile binning, one CTA per 16x16 tile, points staged in
// shared memory as 16-byte (x, y, z, r^2) records, warp-footprint culling by ballot, register top-K.
#include <cfloat>
#include <climits>

#include "binning.cuh"
#include "bulk_copy.cuh"
#include "common.cuh"
#include "raster_math.cuh"

namespace b200r {

constexpr int SETUP_POINTS = 256;
constexpr int PCHUNK = 256;                  // points staged per round (one per thread)
constexpr int QSTRIDE = TILE_THREADS + 1;    // row stride of the per-thread columns in shared memory: slot k of
                                             // thread t lives in bank (k + t) % 32, so neither a warp reading one
                                             // slot nor the row-major write-out of a pixel's K slots conflicts
constexpr int SMEMQ_MAX_K = 32;              // largest K served by the shared-memory queue kernel
constexpr size_t POINT_RECORD_BYTES = 16;    // (x, y, z, radius) per point, written by the setup pass

// Pass 1: per-point box (x +- r, y +- r), skip z < 0 (rasterize_coarse.cu:53-74), count per tile, and the
// 16-byte (x, y, z, r) record the fine pass stages with one vector load.
// The CTA's 256 points (3072 contiguous bytes of the packed (P,3) array) arrive by one TMA bulk copy.
__global__ void __launch_bounds__(SETUP_POINTS)
    points_setup_count_kernel(const float* __restrict__ points, const float* __restrict__ radius, int64_t P,
                              const int64_t* __restrict__ first, const int64_t* __restrict__ num, int N, int H,
                              int W, int TY, int TX, float rx, float ry, uint4* __restrict__ rect,
                              int* __restrict__ tile_count, float4* __restrict__ prec) {
  __shared__ __align__(16) float s_pts[SETUP_POINTS * 3];
  __shared__ __align__(8) uint64_t bar;
  const int tid = threadIdx.x;
  const int64_t p0 = (int64_t)blockIdx.x * SETUP_POINTS;
  const int np = (int)min((int64_t)SETUP_POINTS, P - p0);
  pdl_trigger();  // (see common.cuh: the scan kernel may become resident; it waits for this grid to complete)
  if (tid == 0) {
    mbar_init(&bar, 1);
    fence_mbar_init();
  }
  __syncthreads();
  cta_load_words(s_pts, points + p0 * 3, np * 3, &bar, 0);
  uint2 rc = make_uint2(RECT_EMPTY_X, 0u);
  int n = -1;
  const int64_t pi = p0 + tid;
  if (tid < np) {
    const float x = s_pts[tid * 3 + 0], y = s_pts[tid * 3 + 1], z = s_pts[tid * 3 + 2];  // stride 3: conflict-free
    const float r = __ldg(radius + pi);
    n = find_owner(first, num, N, pi);
    if (n >= 0 && !(z < 0.0f)) rc = bbox_to_tile_rect(fsub(x, r), fadd(x, r), fsub(y, r), fadd(y, r), H, W, rx, ry);
    rect[pi] = make_uint4(rc.x, rc.y, (uint32_t)max(n, 0), 0u);
    prec[pi] = make_float4(x, y, z, r);
  }
  pdl_wait();  // the counters are zeroed by the kernel this one is chained to (see zero_ints_kernel)
  warp_count_rect<false>(rc, n, TY, TX, tile_count, tid & 31);
}

// The same pass with a private per-CTA histogram (see tile_fill_private_kernel in binning.cuh): BIN_CHUNK points per
// CTA, eight per thread, read with plain coalesced loads (consecutive lanes consume consecutive 12-byte points).
__global__ void __launch_bounds__(256)
    points_setup_count_private_kernel(const float* __restrict__ points, const float* __restrict__ radius, int64_t P,
                                      const int64_t* __restrict__ first, const int64_t* __restrict__ num, int N, int H,
                                      int W, int TY, int TX, float rx, float ry, uint4* __restrict__ rect,
                                      int* __restrict__ tile_count, float4* __restrict__ prec) {
  extern __shared__ int hist[];  // [TY * TX]
  const int tid = threadIdx.x, T = TY * TX;
  const int64_t p0 = (int64_t)blockIdx.x * BIN_CHUNK;
  pdl_trigger();
  // all of the thread's points first (one round trip to DRAM for the chunk instead of one per point: the loads were 31 % of
  // the kernel's stall samples when each iteration waited for its own)
  float xs[BIN_CHUNK / 256], ys[BIN_CHUNK / 256], zs[BIN_CHUNK / 256], rs[BIN_CHUNK / 256];
#pragma unroll
  for (int i = 0; i < BIN_CHUNK / 256; ++i) {
    const int64_t pi = p0 + i * 256 + tid;
    xs[i] = ys[i] = zs[i] = rs[i] = 0.0f;
    if (pi < P) {
      xs[i] = __ldg(points + pi * 3 + 0);
      ys[i] = __ldg(points + pi * 3 + 1);
      zs[i] = __ldg(points + pi * 3 + 2);
      rs[i] = __ldg(radius + pi);
    }
  }
  for (int t = tid; t < T; t += 256) hist[t] = 0;
  const int n0 = find_owner(first, num, N, p0);  // the chunk's image (uniform); -1: the chunk starts in a gap
  const int64_t lo0 = n0 >= 0 ? __ldg(first + n0) : 0, hi0 = n0 >= 0 ? lo0 + __ldg(num + n0) : 0;
  __syncthreads();
  pdl_wait();  // the counters are zeroed by the kernel this one is chained to (see zero_ints_kernel)
#pragma unroll
  for (int i = 0; i < BIN_CHUNK / 256; ++i) {
    const int64_t pi = p0 + i * 256 + tid;
    if (pi >= P) continue;
    const float x = xs[i], y = ys[i], z = zs[i], r = rs[i];
    const int n = (pi >= lo0 && pi < hi0) ? n0 : find_owner(first, num, N, pi);
    uint2 rc = make_uint2(RECT_EMPTY_X, 0u);
    if (n >= 0 && !(z < 0.0f)) rc = bbox_to_tile_rect(fsub(x, r), fadd(x, r), fsub(y, r), fadd(y, r), H, W, rx, ry);
    rect[pi] = make_uint4(rc.x, rc.y, (uint32_t)max(n, 0), 0u);
    prec[pi] = make_float4(x, y, z, r);
    if (rect_empty(rc)) continue;
    const int tx0 = rc.x & 0xFFFF, tx1 = rc.x >> 16, ty0 = rc.y & 0xFFFF, ty1 = rc.y >> 16;
    for (int ty = ty0; ty <= ty1; ++ty)
      for (int tx = tx0; tx <= tx1; ++tx) {
        if (n == n0)
          atomicAdd(hist + ty * TX + tx, 1);
        else
          atomicAdd(tile_count + (n * TY + ty) * TX + tx, 1);
      }
  }
  __syncthreads();
  if (n0 >= 0)
    for (int t = tid; t < T; t += 256) {
      const int c = hist[t];
      if (c > 0) atomicAdd(tile_count + n0 * T + t, c);
    }
}

// One staged chunk of points.
struct __align__(16) PointStage {
  union {
    unsigned mask[PCHUNK / 32][TILE_THREADS];         // per pixel (thread): one bit per staged point that covers it
    int sort_buf[2 * TILE_THREADS];                   // exchange buffers of cta_sort256 (before the chunk is staged)
    unsigned long long sort_buf64[2 * TILE_THREADS];  // ... of cta_sort256_u64
  } u;
  float4 rec[PCHUNK];  // x, y, z, r^2 (z < 0: never drawn)
  int id[PCHUNK];
  float col[TILE], row[TILE];  // NDC coordinates of the tile's 16 pixel columns / rows
  int tie;  // points_fine_smem_kernel: some pixel saw a depth tie during an arrival-order walk (flag_point_tie)
};

// (the stage sits at the start of points_fine_smem_kernel's dynamic shared memory: a fixed address, no register)
__device__ __forceinline__ void flag_point_tie() {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  reinterpret_cast<PointStage*>(smem_raw)->tie = 1;
}

struct PointFineParams {
  const float4* prec;  // (x, y, z, r) per point
  const int64_t* first;
  const int64_t* num;
  const int* tile_offset;
  int* pairs;  // tile lists; each CTA puts its own segment in ascending point order before reading it
  int64_t capacity;
  int n0;  // first image of this launch (grid.z is limited to 65535 images)
  int N, H, W, K, TY, TX;
  float rx, ry;
  int smem_ints;  // dynamic shared memory of the launch in 4-byte words (scratch of the in-kernel list sort)
  int vec_ok;     // (W * K) % 4 == 0 and 16-byte aligned outputs: row segments can be written as 16-byte pieces
  int32_t* idx;
  float* zbuf;
  float* dists;
};

__device__ __forceinline__ void stage_point(PointStage& s, int slot, const float4* __restrict__ prec, int pi) {
  const float4 r = __ldg(prec + pi);
  s.rec[slot] = make_float4(r.x, r.y, r.z, fmul(r.w, r.w));
  s.id[slot] = pi;
}

__device__ __forceinline__ void pthread_pixel(int tile_x, int tile_y, int& xo, int& yo) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  xo = tile_x * TILE + (w & 1) * 8 + (lane & 7);
  yo = tile_y * TILE + (w >> 1) * 4 + (lane >> 3);
}

// Thread that owns local pixel (row r, column c) of the tile (inverse of pthread_pixel).
__device__ __forceinline__ int thread_of_pixel(int r, int c) {
  return ((r >> 2) * 2 + (c >> 3)) * 32 + (r & 3) * 8 + (c & 7);
}

// Candidates of one staged chunk.  Every staged point is scan-converted by one thread: the pixels of the tile that can
// lie inside its disc are a small rectangle (pixel_range: the inverse pixel-centre map, a superset), each is tested
// with the reference's arithmetic -- CheckPixelInsidePoint (rasterize_points.cu:49-60): dist2 = fma(dy, dy, rn(dx*dx))
// < rn(r*r), points with z < 0 are skipped -- and a pixel that passes gets the point's bit set in ITS mask
// (mask[point / 32][pixel's thread]).  After one barrier every pixel walks its own mask: its hits, in staging order,
// are offered to `offer(z, point, dist2)` (returns false to stop this pixel's walk).  The search costs ~(pixels in
// the disc's box) per point instead of ~(points in the tile) per pixel: the former box test of every point against
// every warp footprint (one lane per point, a 32x32 bit-matrix transpose per 32 points) was 45 % of the kernel.
// Must be called by the whole CTA; ends with the chunk consumed by this thread (barrier before restaging).
template <class Offer>
__device__ __forceinline__ void points_chunk_scatter_walk(const PointFineParams& p, PointStage& s, int nc, int tile_x,
                                                          int tile_y, bool valid, int lc, int lr, Offer offer) {
  const int tid = threadIdx.x;
  const int nwords = (nc + 31) >> 5;
  // (called after the staging stores and before the barrier that publishes them: the masks are zeroed alongside)
  for (int w = 0; w < nwords; ++w) s.u.mask[w][tid] = 0u;
  __syncthreads();
  if (tid < nc) {
    const float4 r = s.rec[tid];
    if (!(r.z < 0.0f)) {  // points behind the camera are not rendered (rasterize_points.cu:55-56)
      const float rad = sqrtf(r.w) * (1.0f + 1e-6f);  // (r.w = rn(r*r); only the conservative range needs the radius)
      int ix_lo, ix_hi, iy_lo, iy_hi;
      pixel_range(r.x - rad, r.x + rad, p.W, p.rx, ix_lo, ix_hi);
      pixel_range(r.y - rad, r.y + rad, p.H, p.ry, iy_lo, iy_hi);
      // output pixel xo = W - 1 - xi; tile-local column c = xo - tile_x * TILE
      const int c_lo = max(p.W - 1 - ix_hi - tile_x * TILE, 0), c_hi = min(p.W - 1 - ix_lo - tile_x * TILE, TILE - 1);
      const int r_lo = max(p.H - 1 - iy_hi - tile_y * TILE, 0), r_hi = min(p.H - 1 - iy_lo - tile_y * TILE, TILE - 1);
      unsigned* mrow = s.u.mask[tid >> 5];
      const unsigned bit = 1u << (tid & 31);
      for (int rr = r_lo; rr <= r_hi; ++rr) {
        const float dy = fsub(s.row[rr], r.y);
        unsigned* mpix = mrow + (rr >> 2) * 64 + (rr & 3) * 8;  // thread of pixel (rr, c): + (c / 8) * 32 + c % 8
        for (int c = c_lo; c <= c_hi; ++c) {
          const float dx = fsub(s.col[c], r.x);
          if (ffma(dy, dy, fmul(dx, dx)) < r.w) atomicOr(mpix + (c >> 3) * 32 + (c & 7), bit);
        }
      }
    }
  }
  __syncthreads();
  if (!valid) return;
  const float px = s.col[lc], py = s.row[lr];
  int w = 0;
  unsigned m = nwords > 0 ? s.u.mask[0][tid] : 0u;  // (an empty tile has no mask words)
  for (;;) {  // (every lane advances through its own words: see the mesh kernel's walk)
    while (m == 0u && ++w < nwords) m = s.u.mask[w][tid];
    if (m == 0u) break;
    const int j = w * 32 + __ffs((int)m) - 1;
    m &= m - 1u;
    const float4 r = s.rec[j];
    const float dx = fsub(px, r.x), dy = fsub(py, r.y);
    if (!offer(r.z, s.id[j], sqnorm2(dx, dy))) break;
  }
}

// NDC coordinates of the tile's pixel columns and rows (two IEEE divisions each), computed once per tile by 32
// threads; published by the first barrier of the first chunk.
__device__ __forceinline__ void points_tile_coords(const PointFineParams& p, PointStage& s, int tile_x, int tile_y) {
  const int tid = threadIdx.x;
  if (tid < 2 * TILE) {
    const int i = tid & (TILE - 1);
    if (tid < TILE)
      s.col[i] = pix_to_ndc(p.W - 1 - (tile_x * TILE + i), p.W, p.rx);
    else
      s.row[i] = pix_to_ndc(p.H - 1 - (tile_y * TILE + i), p.H, p.ry);
  }
}

// The tile body shared by the point kernels: stage the tile's list chunk by chunk and offer every pixel's hits to
// `offer(z, point, dist2)`.
// `sort_list`: put the tile's list in ascending point order first (the order of the reference's naive kernel,
// rasterize_points.cu:128); without it the points are offered in arrival order (see points_fine_smem_kernel).
// Returns true if the walk was in ascending order (sorted, or an overflowed tile walking the cloud itself).
template <class Offer>
__device__ __forceinline__ bool points_tile_body(const PointFineParams& p, PointStage& s, int* smem_ints_base,
                                                 int tile_x, int tile_y, int n, bool valid, int lc, int lr,
                                                 bool sort_list, Offer offer) {
  const int tid = threadIdx.x;
  pdl_wait();  // the tile lists (fill kernel) and, transitively, the point records are complete (see common.cuh)
  const int tile = (n * p.TY + tile_y) * p.TX + tile_x;
  const int seg_begin = p.tile_offset[tile], seg_end = p.tile_offset[tile + 1];
  const bool overflow = (int64_t)seg_end > p.capacity || seg_end == INT_MAX;
  const int64_t cloud_first = p.first[n];
  const int count = overflow ? (int)p.num[n] : seg_end - seg_begin;
  const bool sort_staged = sort_list && !overflow && count <= PCHUNK;
  if (sort_list && !overflow && count > PCHUNK) {
    cta_sort_segment(p.pairs + seg_begin, count, smem_ints_base, p.smem_ints);
    points_tile_coords(p, s, tile_x, tile_y);  // (the long-list sort may have used the whole stage as scratch)
  }
  for (int base = 0; base < count; base += PCHUNK) {
    const int nc = min(PCHUNK, count - base);
    if (base > 0) __syncthreads();  // previous chunk fully consumed
    int pi = INT_MAX;
    if (tid < nc) pi = overflow ? (int)(cloud_first + base + tid) : p.pairs[seg_begin + base + tid];
    if (sort_staged) {
      pi = cta_sort256(pi, nc, s.u.sort_buf);
      if (nc > 32) __syncthreads();  // the exchange buffers alias the masks zeroed next
    }
    if (tid < nc) stage_point(s, tid, p.prec, pi);
    points_chunk_scatter_walk(p, s, nc, tile_x, tile_y, valid, lc, lr, offer);
  }
  return sort_list || overflow || count <= 1;
}

// Depth-ordered walk of a tile whose list fits one chunk (points_fine_smem_kernel, first attempt).  The CTA sorts the
// tile's points by (z, index) -- one 64-bit key per thread -- and stages them in that order; every pixel then meets its
// hits nearest first, so its K nearest are simply the first K: append-only columns, no eviction, no search for the
// farthest entry, no final sort, and a pixel whose column is full is done.  This equals the reference's result unless two
// of a pixel's hits share a depth bit for bit (their order then depends on the reference's queue history): such a hit
// raises the tile's tie flag and the caller falls back to the literal queue on the index-sorted list.
__device__ __forceinline__ int points_tile_walk_by_depth(const PointFineParams& p, PointStage& s, int seg_begin,
                                                          int count, int tile_x, int tile_y, bool valid, int lc, int lr,
                                                          float* qz, int* qi, float* qd) {
  const int tid = threadIdx.x;
  const int K = p.K;
  unsigned long long key = ~0ull;  // threads without a point, points behind the camera: sorted to the end
  int pi = -1;
  if (tid < count) {
    pi = p.pairs[seg_begin + tid];
    const float z = __ldg(reinterpret_cast<const float*>(p.prec + pi) + 2);
    // (z >= 0: the bits are ordered like the values; -0 + 0 = +0)
    if (!(z < 0.0f)) key = ((unsigned long long)__float_as_uint(fadd(z, 0.0f)) << 32) | (unsigned)pi;
  }
  key = cta_sort256_u64(key, count, s.u.sort_buf64);
  if (count > 32) __syncthreads();  // the exchange buffers alias the masks zeroed next
  if (tid < count) {
    if (key != ~0ull)
      stage_point(s, tid, p.prec, (int)(unsigned)(key & 0xffffffffull));
    else
      s.rec[tid] = make_float4(0.0f, 0.0f, -1.0f, 0.0f);  // (z < 0: never drawn)
  }
  int size = 0;
  float last_z = -1.0f;
  points_chunk_scatter_walk(p, s, count, tile_x, tile_y, valid, lc, lr, [&](float pz, int id, float d2) {
    if (pz == last_z || pz != pz) flag_point_tie();  // equal depths (or NaN): the literal queue decides
    if (size == K) return false;  // the first hit beyond the K nearest: nothing farther can matter
    qz[size * QSTRIDE] = pz;
    qi[size * QSTRIDE] = id;
    qd[size * QSTRIDE] = d2;
    last_z = pz;
    ++size;
    return true;
  });
  return size;
}

// K <= 32: the reference's queue (rasterize_points.cu:61-79) -- an UNSORTED array of K slots plus the tracked
// maximum z; a hit fills the next free slot or, when full and pz < q_max_z, overwrites the tracked maximum,
// which is then searched again -- with its three arrays in dynamic shared memory as per-thread columns, where
// the dynamic slot index costs nothing.  Points arrive in ascending index order (sorted tile lists), so tie
// behaviour equals the reference's naive kernel.  The epilogue sorts each column (stable, on z only) and the CTA
// writes the tile's outputs row segment by row segment: 16 pixels x K values are contiguous in memory, so every
// store instruction fills whole 32-byte sectors (per-pixel stores at a 4*K-byte stride filled one eighth).
__global__ void __launch_bounds__(TILE_THREADS) points_fine_smem_kernel(const PointFineParams p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  PointStage& s = *reinterpret_cast<PointStage*>(smem_raw);
  const int tid = threadIdx.x;
  const int K = p.K;
  float* qz0 = reinterpret_cast<float*>(smem_raw + sizeof(PointStage));
  int* qi0 = reinterpret_cast<int*>(qz0 + K * QSTRIDE);
  float* qd0 = reinterpret_cast<float*>(qi0 + K * QSTRIDE);
  float* qz = qz0 + tid;  // qz[k * QSTRIDE]
  int* qi = qi0 + tid;
  float* qd = qd0 + tid;
  const int tile_x = blockIdx.x, tile_y = blockIdx.y, n = p.n0 + blockIdx.z;
  const int tile = (n * p.TY + tile_y) * p.TX + tile_x;
  int xo, yo;
  pthread_pixel(tile_x, tile_y, xo, yo);
  const bool valid = xo < p.W && yo < p.H;
  const int lc = xo - tile_x * TILE, lr = yo - tile_y * TILE;  // local column / row of my pixel
  points_tile_coords(p, s, tile_x, tile_y);
  pdl_wait();  // the tile lists (fill kernel) and, transitively, the point records are complete (see common.cuh)

  // Order of the list: the queue keeps the K nearest points whatever the arrival order unless two points share,
  // bit for bit, the depth at the queue's far end, and the final stable sort on z orders them the same way unless two
  // kept points share a depth.  Point depths rarely tie, so the tile is first walked in arrival order while
  // watching for exactly those events; only if some pixel saw one is the list sorted (ascending point index, the
  // order of the reference's naive kernel) and the tile walked again.
  // A list that fits one chunk (all but very dense tiles) is first walked in DEPTH order (points_tile_walk_by_depth),
  // which needs neither the queue's eviction logic nor a final sort; it is equally exact unless depths tie.
  int size, max_idx;
  float max_z;
  const int seg_begin0 = p.tile_offset[tile], seg_end0 = p.tile_offset[tile + 1];
  const bool by_depth_ok = !((int64_t)seg_end0 > p.capacity || seg_end0 == INT_MAX) && seg_end0 - seg_begin0 <= PCHUNK;
  for (int attempt = by_depth_ok ? 0 : 1;; attempt = 2) {  // 0: depth order, 1: arrival order, 2: index order (exact)
    const bool sort_list = attempt == 2;
    size = 0;
    max_idx = -1;
    max_z = -1000.0f;
    if (tid == 0 && !sort_list) s.tie = 0;  // (ordered before every offer by the barriers of the tile body)
    if (attempt == 0) {
      size = points_tile_walk_by_depth(p, s, seg_begin0, seg_end0 - seg_begin0, tile_x, tile_y, valid, lc, lr, qz, qi,
                                       qd);
      if (!p.vec_ok) {
        if (__syncthreads_or(s.tie)) continue;
        if (!valid) return;
        const int64_t o = (((int64_t)n * p.H + yo) * p.W + xo) * K;
        for (int k = 0; k < K; ++k) {
          const bool e = k >= size;
          p.idx[o + k] = e ? -1 : qi[k * QSTRIDE];
          p.zbuf[o + k] = e ? -1.0f : qz[k * QSTRIDE];
          p.dists[o + k] = e ? -1.0f : qd[k * QSTRIDE];
        }
        return;
      }
      for (int k = size; k < K; ++k) {  // the -1 padding of the unused slots
        qz[k * QSTRIDE] = -1.0f;
        qi[k * QSTRIDE] = -1;
        qd[k * QSTRIDE] = -1.0f;
      }
      if (!__syncthreads_or(s.tie)) break;  // no depth tie anywhere: the depth-order walk stands
      continue;
    }
    const bool in_order = points_tile_body(
        p, s, reinterpret_cast<int*>(smem_raw), tile_x, tile_y, n, valid, lc, lr, sort_list,
        [&](float pz, int pi, float d2) {
          if (size < K) {  // (:61-67)
            qz[size * QSTRIDE] = pz;
            qi[size * QSTRIDE] = pi;
            qd[size * QSTRIDE] = d2;
            if (pz > max_z) {
              max_z = pz;
              max_idx = size;
            }
            ++size;
          } else if (pz < max_z) {  // (:68-78)
            const float evicted = max_z;
            qz[max_idx * QSTRIDE] = pz;
            qi[max_idx * QSTRIDE] = pi;
            qd[max_idx * QSTRIDE] = d2;
            max_z = pz;
            for (int i = 0; i < K; ++i) {
              const float v = qz[i * QSTRIDE];
              if (v > max_z) {
                max_z = v;
                max_idx = i;
              }
            }
            if (max_z == evicted) flag_point_tie();
          } else if (pz == max_z) {
            flag_point_tie();
          }
          return true;
        });
    // BubbleSort on z only (rasterize_points.cu:26-28): stable -> insertion sort over the thread's own column
    for (int i = 1; i < size; ++i) {
      const float tz = qz[i * QSTRIDE], td = qd[i * QSTRIDE];
      const int ti = qi[i * QSTRIDE];
      int j = i - 1;
      while (j >= 0 && tz < qz[j * QSTRIDE]) {
        qz[(j + 1) * QSTRIDE] = qz[j * QSTRIDE];
        qi[(j + 1) * QSTRIDE] = qi[j * QSTRIDE];
        qd[(j + 1) * QSTRIDE] = qd[j * QSTRIDE];
        --j;
      }
      if (j >= 0 && tz == qz[j * QSTRIDE]) flag_point_tie();  // equal depths keep their arrival order
      qz[(j + 1) * QSTRIDE] = tz;
      qi[(j + 1) * QSTRIDE] = ti;
      qd[(j + 1) * QSTRIDE] = td;
    }
    if (!p.vec_ok) {
      // (CTA-uniform) did any pixel see a tie?  then walk again, sorted, before anything is written.  Every thread
      // contributes its own view of the flag: the thread that raised it sees it, and nobody reads it after the barrier
      if (!in_order && __syncthreads_or(s.tie)) continue;
      if (!valid) return;
      const int64_t o = (((int64_t)n * p.H + yo) * p.W + xo) * K;
      for (int k = 0; k < K; ++k) {
        const bool e = k >= size;
        p.idx[o + k] = e ? -1 : qi[k * QSTRIDE];
        p.zbuf[o + k] = e ? -1.0f : qz[k * QSTRIDE];
        p.dists[o + k] = e ? -1.0f : qd[k * QSTRIDE];
      }
      return;
    }
    for (int k = size; k < K; ++k) {  // the -1 padding of the unused slots
      qz[k * QSTRIDE] = -1.0f;
      qi[k * QSTRIDE] = -1;
      qd[k * QSTRIDE] = -1.0f;
    }
    // (barrier: the columns are complete; OR of every thread's view of the flag, which nobody reads afterwards)
    if (!__syncthreads_or(in_order ? 0 : s.tie)) break;  // no depth tie anywhere: the arrival-order walk stands
  }
  // row-major write-out: row r of the tile is npx * K consecutive values of each output
  const int x0 = tile_x * TILE, y0 = tile_y * TILE;
  const int npx = min(TILE, p.W - x0), nrow = min(TILE, p.H - y0);
  const int seg4 = (npx * K) >> 2;  // 16-byte pieces per row segment (npx * K is a multiple of 4 when vec_ok)
  for (int e = tid; e < nrow * seg4; e += TILE_THREADS) {
    const int r = e / seg4, v = e - r * seg4;
    int c = (4 * v) / K, k = 4 * v - c * K;
    float z[4], d[4];
    int id[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int at = k * QSTRIDE + thread_of_pixel(r, c);
      z[j] = qz0[at];
      id[j] = qi0[at];
      d[j] = qd0[at];
      if (++k == K) {
        k = 0;
        ++c;
      }
    }
    const int64_t o4 = (((((int64_t)n * p.H + y0 + r) * p.W + x0) * K) >> 2) + v;
    __stcs(reinterpret_cast<int4*>(p.idx) + o4, make_int4(id[0], id[1], id[2], id[3]));
    __stcs(reinterpret_cast<float4*>(p.zbuf) + o4, make_float4(z[0], z[1], z[2], z[3]));
    __stcs(reinterpret_cast<float4*>(p.dists) + o4, make_float4(d[0], d[1], d[2], d[3]));
  }
}

// 32 < K <= 150: the same queue in thread-local arrays.
__global__ void __launch_bounds__(TILE_THREADS) points_fine_bigk_kernel(const PointFineParams p) {
  __shared__ PointStage s;
  const int K = p.K;
  const int tile_x = blockIdx.x, tile_y = blockIdx.y, n = p.n0 + blockIdx.z;
  int xo, yo;
  pthread_pixel(tile_x, tile_y, xo, yo);
  const bool valid = xo < p.W && yo < p.H;
  const int lc = xo - tile_x * TILE, lr = yo - tile_y * TILE;
  points_tile_coords(p, s, tile_x, tile_y);
  float lz[B200R_MAX_K], ld[B200R_MAX_K];
  int li[B200R_MAX_K];
  int ln = 0, l_max_idx = -1;
  float l_max_z = -1000.0f;
  points_tile_body(p, s, reinterpret_cast<int*>(&s), tile_x, tile_y, n, valid, lc, lr, true,
                   [&](float pz, int pi, float d2) {
    if (ln < K) {
      lz[ln] = pz;
      li[ln] = pi;
      ld[ln] = d2;
      if (pz > l_max_z) {
        l_max_z = pz;
        l_max_idx = ln;
      }
      ++ln;
    } else if (pz < l_max_z) {
      lz[l_max_idx] = pz;
      li[l_max_idx] = pi;
      ld[l_max_idx] = d2;
      l_max_z = pz;
      for (int i = 0; i < K; ++i)
        if (lz[i] > l_max_z) {
          l_max_z = lz[i];
          l_max_idx = i;
        }
    }
    return true;
  });
  if (!valid) return;
  for (int i = 1; i < ln; ++i) {  // stable insertion sort on z only
    const float tz = lz[i], td = ld[i];
    const int ti = li[i];
    int j = i - 1;
    while (j >= 0 && tz < lz[j]) {
      lz[j + 1] = lz[j];
      li[j + 1] = li[j];
      ld[j + 1] = ld[j];
      --j;
    }
    lz[j + 1] = tz;
    li[j + 1] = ti;
    ld[j + 1] = td;
  }
  const int64_t o = (((int64_t)n * p.H + yo) * p.W + xo) * K;
  for (int k = 0; k < K; ++k) {
    p.idx[o + k] = k < ln ? li[k] : -1;
    p.zbuf[o + k] = k < ln ? lz[k] : -1.0f;
    p.dists[o + k] = k < ln ? ld[k] : -1.0f;
  }
}

// Backward (rasterize_points.cu:366-411): grad_xy = 2 * grad_dist * (p_xy - pix_xy), grad_z = grad_zbuf.
// One thread per pixel on the forward pass's tiles and 8x4 footprints, looping over the K slots.  A point covers
// many neighbouring pixels, so at every slot the warp first merges ALL lanes that hold the same point
// (__match_any_sync + pointer jumping, as in the mesh backward) and only one lane per distinct point issues the
// three atomics.  STAGED: the tile's indices and upstream gradients are first read row segment by row segment
// (16 pixels x K values are contiguous: coalesced 16-byte loads) into per-thread columns in shared memory;
// otherwise (K > 32, or rows that are not 16-byte multiples) every thread reads its own K values directly.
template <bool STAGED>
__global__ void __launch_bounds__(TILE_THREADS)
    points_backward_kernel(const float* __restrict__ points, const int32_t* __restrict__ idxs,
                           const float* __restrict__ grad_zbuf, const float* __restrict__ grad_dists, int n0, int H,
                           int W, int K, float rx, float ry, float* __restrict__ grad_points, int g_vec) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int tid = threadIdx.x, lane = tid & 31;
  const int tile_x = blockIdx.x, tile_y = blockIdx.y, n = n0 + blockIdx.z;
  int xo, yo;
  pthread_pixel(tile_x, tile_y, xo, yo);
  const bool in_image = xo < W && yo < H;
  const float xf = pix_to_ndc(W - 1 - xo, W, rx);
  const float yf = pix_to_ndc(H - 1 - yo, H, ry);
  const int64_t o = in_image ? (((int64_t)n * H + yo) * W + xo) * K : 0;
  int* si0 = reinterpret_cast<int*>(smem_raw);
  float* sz0 = reinterpret_cast<float*>(si0 + K * QSTRIDE);
  float* sd0 = sz0 + K * QSTRIDE;
  if (STAGED) {
    const int x0 = tile_x * TILE, y0 = tile_y * TILE;
    const int npx = min(TILE, W - x0), nrow = min(TILE, H - y0);
    const int seg4 = (npx * K) >> 2;
    for (int e = tid; e < nrow * seg4; e += TILE_THREADS) {
      const int r = e / seg4, v = e - r * seg4;
      const int64_t o4 = (((((int64_t)n * H + y0 + r) * W + x0) * K) >> 2) + v;
      const int4 vi = __ldcs(reinterpret_cast<const int4*>(idxs) + o4);
      const float4 vz = __ldcs(reinterpret_cast<const float4*>(grad_zbuf) + o4);
      const float4 vd = __ldcs(reinterpret_cast<const float4*>(grad_dists) + o4);
      const int ii[4] = {vi.x, vi.y, vi.z, vi.w};
      const float zz[4] = {vz.x, vz.y, vz.z, vz.w}, dd[4] = {vd.x, vd.y, vd.z, vd.w};
      int c = (4 * v) / K, k = 4 * v - c * K;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int at = k * QSTRIDE + thread_of_pixel(r, c);
        si0[at] = ii[j];
        sz0[at] = zz[j];
        sd0[at] = dd[j];
        if (++k == K) {
          k = 0;
          ++c;
        }
      }
    }
    __syncthreads();
  }
  for (int k = 0; k < K; ++k) {
    int pi = -1;
    if (in_image) pi = STAGED ? si0[k * QSTRIDE + tid] : idxs[o + k];
    if (!__any_sync(0xffffffffu, pi >= 0)) continue;
    float gx = 0.0f, gy = 0.0f, gz = 0.0f;
    if (pi >= 0) {
      const float gd = STAGED ? sd0[k * QSTRIDE + tid] : grad_dists[o + k];
      const float g2 = gd + gd;
      gx = g2 * (__ldg(points + (int64_t)pi * 3 + 0) - xf);
      gy = g2 * (__ldg(points + (int64_t)pi * 3 + 1) - yf);
      gz = STAGED ? sz0[k * QSTRIDE + tid] : grad_zbuf[o + k];
    }
    const unsigned grp = __match_any_sync(0xffffffffu, pi);
    const unsigned above = lane == 31 ? 0u : grp & (0xffffffffu << (lane + 1));
    int next = (pi >= 0 && above != 0u) ? __ffs((int)above) - 1 : -1;
    while (__any_sync(0xffffffffu, next >= 0)) {
      const int src = next >= 0 ? next : lane;
      const float vx = __shfl_sync(0xffffffffu, gx, src), vy = __shfl_sync(0xffffffffu, gy, src),
                  vz = __shfl_sync(0xffffffffu, gz, src);
      const int nn = __shfl_sync(0xffffffffu, next, src);
      if (next >= 0) {
        gx += vx;
        gy += vy;
        gz += vz;
      }
      next = next >= 0 ? nn : -1;
    }
    if (pi >= 0 && lane == __ffs((int)grp) - 1) {
      float* o = grad_points + (int64_t)pi * 3;
      if (g_vec) {
        // (a point's 12 bytes start at a multiple of 4 whose parity is that of the index: one 8-byte vector reduction and
        // one scalar one instead of three -- fewer instructions through the L1 / MIO pipeline, the same sums)
        const bool odd = (pi & 1) != 0;
        atomicAdd(o + (odd ? 0 : 2), odd ? gx : gz);
        asm volatile("red.global.add.v2.f32 [%0], {%1, %2};" ::"l"(o + (odd ? 1 : 0)), "f"(odd ? gy : gx), "f"(odd ? gz : gy)
                     : "memory");
      } else {
        atomicAdd(o + 0, gx);
        atomicAdd(o + 1, gy);
        atomicAdd(o + 2, gz);
      }
    }
  }
}

}  // namespace b200r

using namespace b200r;

extern "C" size_t b200r_rasterize_points_workspace_bytes(int64_t P, int32_t N, int32_t H, int32_t W,
                                                         int64_t pair_capacity) {
  if (P < 0 || N < 0 || H < 0 || W < 0) return 0;
  return carve_workspace(nullptr, P, N, H, W, pair_capacity).bytes + POINT_RECORD_BYTES * (size_t)(P > 0 ? P : 1);
}

static bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

extern "C" int b200r_rasterize_points_forward(const float* points, int64_t P, const int64_t* first,
                                              const int64_t* num, const float* radius, int32_t N, int32_t H,
                                              int32_t W, int32_t K, int32_t bin_size, int32_t max_points_per_bin,
                                              int32_t* idx, float* zbuf, float* dists, void* workspace,
                                              size_t workspace_bytes, int64_t pair_capacity, void* stream_) {
  (void)bin_size;
  (void)max_points_per_bin;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  if (K > B200R_MAX_K) return fail(B200R_ERR_INVALID_ARGUMENT, "Must have num_closest <= 150");
  if (P < 0 || N < 0 || H < 0 || W < 0 || K < 0) return fail(B200R_ERR_INVALID_ARGUMENT, "negative size");
  if (P > INT_MAX) return fail(B200R_ERR_INVALID_ARGUMENT, "more than 2^31-1 packed points are not supported");
  if ((int64_t)N * H * W * K == 0) return B200R_OK;
  const int TY = div_up(H, TILE), TX = div_up(W, TILE);
  if (TY > 0xFFFE || TX > 0xFFFE) return fail(B200R_ERR_INVALID_ARGUMENT, "image too large");
  const int64_t ntiles = (int64_t)N * TY * TX;
  if (ntiles > INT_MAX) return fail(B200R_ERR_INVALID_ARGUMENT, "too many tiles");
  BinWorkspace ws = carve_workspace(workspace, P, N, H, W, pair_capacity);
  const size_t nrec = (size_t)(P > 0 ? P : 1);
  if (workspace == nullptr || workspace_bytes < ws.bytes + POINT_RECORD_BYTES * nrec)
    return fail(B200R_ERR_WORKSPACE, "workspace too small for rasterize_points_forward");
  float4* prec = reinterpret_cast<float4*>(static_cast<char*>(workspace) + ws.bytes);  // (ws.bytes % 16 == 0)
  const float rx = ndc_range(W, H), ry = ndc_range(H, W);

  const bool prof = profiling_enabled();
  if (prof) phase_timer().record(0, stream);
  zero_ints_kernel<<<(unsigned)((ntiles + 1023) / 1024), 256, 0, stream>>>(ws.tile_count, ntiles);
  B200R_LAUNCHED("zero_ints_kernel");
  // (a private histogram over one image's tiles per CTA, if it fits; see binning.cuh)
  const bool private_hist = (int64_t)TY * TX <= BIN_MAX_TILES;
  const size_t hist_bytes = sizeof(int) * (size_t)TY * TX;
  if (P > 0) {
    // (chained to the zeroing kernel: the loads and the per-point arithmetic overlap it)
    if (private_hist)
      B200R_CUDA_OK(launch_chained(points_setup_count_private_kernel, dim3((unsigned)((P + BIN_CHUNK - 1) / BIN_CHUNK)),
                                   dim3(256), hist_bytes, stream, points, radius, P, first, num, N, H, W, TY, TX, rx, ry,
                                   ws.rect, ws.tile_count, prec));
    else
      B200R_CUDA_OK(launch_chained(points_setup_count_kernel, dim3((unsigned)((P + SETUP_POINTS - 1) / SETUP_POINTS)),
                                   dim3(SETUP_POINTS), 0, stream, points, radius, P, first, num, N, H, W, TY, TX, rx, ry,
                                   ws.rect, ws.tile_count, prec));
    B200R_LAUNCHED("points_setup_count_kernel");
  }
  B200R_CUDA_OK(launch_chained(tile_scan_kernel, dim3(1), dim3(1024), 0, stream, ws.tile_count, ws.tile_offset,
                               (int)ntiles, (int*)nullptr));
  B200R_LAUNCHED("tile_scan_kernel");
  if (P > 0) {
    if (private_hist)
      B200R_CUDA_OK(launch_chained(tile_fill_private_kernel, dim3((unsigned)((P + BIN_CHUNK - 1) / BIN_CHUNK)), dim3(256),
                                   hist_bytes, stream, ws.rect, P, TY, TX, ws.tile_count, ws.pairs, ws.capacity));
    else
      B200R_CUDA_OK(launch_chained(tile_fill_kernel<false>, dim3((unsigned)((P + 255) / 256)), dim3(256), 0, stream,
                                   ws.rect, P, TY, TX, ws.tile_count, ws.pairs, ws.capacity));
    B200R_LAUNCHED("tile_fill_kernel");
  }
  // (no sort launch: every fine CTA puts its own tile list in ascending point order, see cta_sort256)
  if (prof) phase_timer().record(1, stream);
  PointFineParams p;
  p.prec = prec; p.first = first; p.num = num;
  p.tile_offset = ws.tile_offset; p.pairs = ws.pairs; p.capacity = ws.capacity;
  p.N = N; p.H = H; p.W = W; p.K = K; p.TY = TY; p.TX = TX; p.rx = rx; p.ry = ry;
  p.idx = idx; p.zbuf = zbuf; p.dists = dists;
  p.vec_ok = (((int64_t)W * K) % 4 == 0 && aligned16(idx) && aligned16(zbuf) && aligned16(dists)) ? 1 : 0;
  size_t smem = 0;
  if (K <= SMEMQ_MAX_K) {
    smem = sizeof(PointStage) + (size_t)K * QSTRIDE * 12;
    static bool configured[64] = {}; /* > 48 KB of dynamic shared memory: opt-in per kernel and device */
    int dev_ = 0;
    B200R_CUDA_OK(cudaGetDevice(&dev_));
    if (dev_ < 0 || dev_ >= 64 || !configured[dev_]) {
      B200R_CUDA_OK(cudaFuncSetAttribute(points_fine_smem_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)(sizeof(PointStage) + (size_t)SMEMQ_MAX_K * QSTRIDE * 12)));
      if (dev_ >= 0 && dev_ < 64) configured[dev_] = true;
    }
    p.smem_ints = (int)(smem / sizeof(int));
  } else {
    p.smem_ints = (int)(sizeof(PointStage) / sizeof(int));
  }
  for (p.n0 = 0; p.n0 < N; p.n0 += 65535) {  // grid.z is limited to 65535 images per launch
    const dim3 grid3((unsigned)TX, (unsigned)TY, (unsigned)min(N - p.n0, 65535));
    if (K <= SMEMQ_MAX_K)
      B200R_CUDA_OK(launch_chained(points_fine_smem_kernel, grid3, dim3(TILE_THREADS), smem, stream, p));
    else
      B200R_CUDA_OK(launch_chained(points_fine_bigk_kernel, grid3, dim3(TILE_THREADS), 0, stream, p));
  }
  B200R_LAUNCHED("points_fine_kernel");
  if (prof) {
    phase_timer().record(2, stream);
    phase_timer().have_fwd = true;
  }
  return B200R_OK;
}

extern "C" int b200r_rasterize_points_backward(const float* points, int64_t P, const int32_t* idxs,
                                               const float* grad_zbuf, const float* grad_dists, int32_t N,
                                               int32_t H, int32_t W, int32_t K, float* grad_points, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  if (P < 0 || N < 0 || H < 0 || W < 0 || K < 0) return fail(B200R_ERR_INVALID_ARGUMENT, "negative size");
  if (P == 0) return B200R_OK;
  B200R_CUDA_OK(cudaMemsetAsync(grad_points, 0, sizeof(float) * 3 * (size_t)P, stream));
  const int64_t total = (int64_t)N * H * W * K;
  if (total == 0) return B200R_OK;
  const int TY = div_up(H, TILE), TX = div_up(W, TILE);
  if (TY > 65535) return fail(B200R_ERR_INVALID_ARGUMENT, "image too large");
  const bool prof = profiling_enabled();
  if (prof) phase_timer().record(3, stream);
  const bool staged = K <= SMEMQ_MAX_K && ((int64_t)W * K) % 4 == 0 && aligned16(idxs) && aligned16(grad_zbuf) &&
                      aligned16(grad_dists);
  const size_t smem = staged ? (size_t)K * QSTRIDE * 12 : 0;
  const int g_vec = (reinterpret_cast<uintptr_t>(grad_points) & 7u) == 0 ? 1 : 0;
  if (staged) {
    static bool configured[64] = {};
    int dev_ = 0;
    B200R_CUDA_OK(cudaGetDevice(&dev_));
    if (dev_ < 0 || dev_ >= 64 || !configured[dev_]) {
      B200R_CUDA_OK(cudaFuncSetAttribute(points_backward_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)((size_t)SMEMQ_MAX_K * QSTRIDE * 12)));
      if (dev_ >= 0 && dev_ < 64) configured[dev_] = true;
    }
  }
  for (int n0 = 0; n0 < N; n0 += 65535) {  // grid.z is limited to 65535 images per launch
    const dim3 grid((unsigned)TX, (unsigned)TY, (unsigned)min(N - n0, 65535));
    if (staged)
      points_backward_kernel<true><<<grid, TILE_THREADS, smem, stream>>>(points, idxs, grad_zbuf, grad_dists, n0, H,
                                                                       W, K, ndc_range(W, H), ndc_range(H, W),
                                                                       grad_points, g_vec);
    else
      points_backward_kernel<false><<<grid, TILE_THREADS, 0, stream>>>(points, idxs, grad_zbuf, grad_dists, n0, H,
                                                                       W, K, ndc_range(W, H), ndc_range(H, W),
                                                                       grad_points, g_vec);
  }
  B200R_LAUNCHED("points_backward_kernel");
  if (prof) {
    phase_timer().record(4, stream);
    phase_timer().have_bwd = true;
  }
  return B200R_OK;
}
