// Mesh rasterizer for sm_100a: setup/bin pass, per-tile fine pass (top-K per pixel), backward.
//
// Replaces, behind the same operator signature, the reference's
//   TriangleBoundingBoxKernel + RasterizeCoarseCudaKernel   (rasterize_coarse.cu:20-51, 76-219)
//   RasterizeMeshesFineCudaKernel / RasterizeMeshesNaiveCudaKernel (rasterize_meshes.cu:630-736, 245-334)
//   RasterizeMeshesBackwardCudaKernel                        (rasterize_meshes.cu:433-564)
// Design (see DESIGN.md): exact tile binning (binning.cuh); the setup pass also writes a 64-byte record per
// face (vertices, barycentric denominator, exact pixel rectangle or blur-expanded box).  One CTA per 16x16 pixel
// tile gathers the records of the tile's faces into shared memory; each warp owns an 8x4 pixel footprint.
// Without blur the faces are scan-converted into per-pixel candidate bitmasks (division-free inside test), with
// blur each lane box-tests one face against the footprint and a warp bit-matrix transpose yields per-pixel
// masks; the exact per-pixel arithmetic of raster_math.cuh runs only on candidates, in ascending face order.
// The K nearest hits are the reference's queue: keys in registers, payload in shared memory.
#include <cfloat>
#include <climits>

#include "binning.cuh"
#include "bulk_copy.cuh"
#include "common.cuh"
#include "raster_math.cuh"

namespace b200r {

constexpr int SETUP_FACES = 256;  // faces per CTA in the setup pass (one per thread)
// Tile of the mesh FORWARD pass (binning + fine kernels): FTW x FTH pixels, one thread per pixel, warps own 8x4
// footprints.  (The backward kernels and the point rasterizer keep TILE x TILE = 16 x 16.)
// (16 x 8 tiles were measured: north-star fine 141.3 -> 141.9 us, binning 45 -> 51 us, config 5 9.3 -> 10.3 ms; only
// config 2 gains, 139.7 -> 123.4 us.)
constexpr int FTW = 16, FTH = 16, FTHREADS = FTW * FTH;
static_assert(FTH == 16 || FTH == 8, "16x16 or 16x8 tiles");
constexpr int CHUNK = FTHREADS;   // faces staged per round in the fine pass (one per thread)
constexpr int SMEMQ_MAX_K = 32;   // largest K served by the shared-memory queue kernel (mesh_fine_smemq_kernel)

// ------------------------------------------------------------------------------------------------
// Pass 1: per-face validity + blur-expanded box -> tile rectangle, count per tile.
// The CTA's 256 faces (9216 contiguous bytes of the packed (F,3,3) array) arrive by one TMA bulk copy.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ bool face_is_drawable(const Face& f, bool cull_backfaces) {
  const float zmax = fmaxf(fmaxf(f.z0, f.z1), f.z2), zmin = fminf(fminf(f.z0, f.z1), f.z2);
  if (!(zmax >= 0.0f)) return false;           // behind the camera            (rasterize_meshes.cu:138,147)
  if ((double)zmin < kEps) return false;       // z_invalid (double compare)   (:92)
  const float area = edge_fn(f.x0, f.y0, f.x1, f.y1, f.x2, f.y2);  // EdgeFunctionForward(v0, v1, v2) (:141)
  if (cull_backfaces && area < 0.0f) return false;                  // (:143,147)
  if ((double)fabsf(area) <= kEps) return false;                    // zero_face_area (:144-145)
  return true;
}

__device__ __forceinline__ void face_box(const Face& f, float sqrt_blur, float& xmin, float& xmax, float& ymin,
                                         float& ymax) {
  xmin = fsub(fminf(fminf(f.x0, f.x1), f.x2), sqrt_blur);  // (:85-88)
  xmax = fadd(fmaxf(fmaxf(f.x0, f.x1), f.x2), sqrt_blur);
  ymin = fsub(fminf(fminf(f.y0, f.y1), f.y2), sqrt_blur);
  ymax = fadd(fmaxf(fmaxf(f.y0, f.y1), f.y2), sqrt_blur);
}

// Per-face records (workspace, written once per forward call by the setup pass, gathered by the fine pass): the
// constants of a face that every (tile, face) pair would otherwise recompute.  Four 16-byte words per face:
//   [0] x0, y0, x1, y1
//   [1] x2, y2, barycentric denominator, face index (int bits)
//   [2] z0, z1, z2, clipped-face neighbour index (int bits, -1 = none)
//   [3] blur_radius == 0: xo_lo, xo_hi, yo_lo, yo_hi (int): the OUTPUT pixels whose centre passes the reference's
//       box test;  blur_radius > 0: xmin, xmax, ymin, ymax of the blur-expanded box (empty = never hit)
constexpr size_t FACE_RECORD_BYTES = 4 * 16;

// Exact pixel range of the box test `p > vmax || p < vmin` (rasterize_meshes.cu:94-97): pix_to_ndc is monotonic
// in the pixel index, so the passing pixels are contiguous.  The inverse pixel-centre map in plain float locates
// each end to within `margin` pixels (see pixel_range); if no pixel centre lies that close to the end, the rounded
// index is already exact (all but ~0.2 % of the ends), otherwise the end is settled by evaluating pix_to_ndc
// itself -- two IEEE divisions that the common case never executes.
__device__ __forceinline__ void exact_pixel_range(float vmin, float vmax, int S, float range, int& lo, int& hi) {
  const float off = range * 0.5f, scale = (float)S / range, margin = 1e-3f + 1e-6f * (float)S;
  const float a = (vmin + off) * scale - 0.5f, b = (vmax + off) * scale - 0.5f;
  // conservative ends (identical to pixel_range) and the ends if the map erred the other way
  const float a0 = fminf(fmaxf(a - margin, -1.0f), (float)S + 1.0f), a1 = fminf(fmaxf(a + margin, -1.0f), (float)S + 1.0f);
  const float b0 = fminf(fmaxf(b + margin, -2.0f), (float)S), b1 = fminf(fmaxf(b - margin, -2.0f), (float)S);
  lo = max(0, (int)ceilf(a0));
  hi = min(S - 1, (int)floorf(b0));
  const bool lo_sure = lo == max(0, (int)ceilf(a1)) && a == a;  // (a != a: NaN coordinates take the slow path)
  const bool hi_sure = hi == min(S - 1, (int)floorf(b1)) && b == b;
  if (!lo_sure) {
    while (lo <= hi) {
      const float v = pix_to_ndc(lo, S, range);
      if (!(v > vmax || v < vmin)) break;
      ++lo;
    }
  }
  if (!hi_sure) {
    while (hi >= lo) {
      const float v = pix_to_ndc(hi, S, range);
      if (!(v > vmax || v < vmin)) break;
      --hi;
    }
  }
}

// INDEXED (the fused entry point): the faces are given as (verts, faces); the kernel gathers the three vertices
// of each face itself -- what `verts_packed[faces_packed]` does in the reference's wrapper
// (rasterize_meshes.py:144-148) -- and also writes the gathered (F,3,3) array for the backward pass.
// Resident CTAs per SM the register budget is set for (6 / 8: binning 44.8 -> 45.6 / 46.8 us).
constexpr int SETUP_CTAS = 1;
template <bool INDEXED>
__global__ void __launch_bounds__(SETUP_FACES, SETUP_CTAS)
    mesh_setup_count_kernel(const float* __restrict__ face_verts, const float* __restrict__ verts, int64_t V,
                            const int64_t* __restrict__ faces, float* __restrict__ face_verts_out,
                            const int64_t* __restrict__ neighbor, int64_t F, const int64_t* __restrict__ first,
                            const int64_t* __restrict__ num, int N, int H, int W, int TY, int TX, float rx, float ry,
                            float sqrt_blur, int cull_backfaces, uint4* __restrict__ rect,
                            int* __restrict__ tile_count, float4* __restrict__ rec) {
  __shared__ __align__(16) float s_fv[SETUP_FACES * 9];
  __shared__ __align__(8) uint64_t bar;
  const int tid = threadIdx.x;
  const int64_t f0 = (int64_t)blockIdx.x * SETUP_FACES;
  const int nf = (int)min((int64_t)SETUP_FACES, F - f0);
  pdl_trigger();  // (see common.cuh: the scan kernel may become resident; it waits for this grid to complete)
  if (INDEXED) {
    // one (face, corner) per step and thread: coalesced index reads, 12-byte vertex gathers (the vertex array
    // is small and L2-resident), then the gathered block is written out as 9 * nf contiguous floats
    for (int e = tid; e < nf * 3; e += SETUP_FACES) {
      const int64_t vi = __ldg(faces + f0 * 3 + e);
      const bool ok = vi >= 0 && vi < V;  // out-of-range indices (an error in the reference) give a NaN face
      const float* v = verts + vi * 3;
      s_fv[e * 3 + 0] = ok ? __ldg(v + 0) : __int_as_float(0x7fc00000);
      s_fv[e * 3 + 1] = ok ? __ldg(v + 1) : __int_as_float(0x7fc00000);
      s_fv[e * 3 + 2] = ok ? __ldg(v + 2) : __int_as_float(0x7fc00000);
    }
    __syncthreads();
    for (int e = tid; e < nf * 9; e += SETUP_FACES) face_verts_out[f0 * 9 + e] = s_fv[e];
  } else {
    if (tid == 0) {
      mbar_init(&bar, 1);
      fence_mbar_init();
    }
    __syncthreads();
    cta_load_words(s_fv, face_verts + f0 * 9, nf * 9, &bar, 0);
  }
  uint2 r = make_uint2(RECT_EMPTY_X, 0u);
  int n = -1;
  const int64_t fi = f0 + tid;
  if (tid < nf) {
    const float* v = s_fv + tid * 9;  // stride 9 words: conflict-free across a warp
    const Face f = {v[0], v[1], v[2], v[3], v[4], v[5], v[6], v[7], v[8]};
    n = find_owner(first, num, N, fi);
    float4 box = make_float4(FLT_MAX, -FLT_MAX, FLT_MAX, -FLT_MAX);
    int4 rng = make_int4(1, 0, 1, 0);
    if (n >= 0 && face_is_drawable(f, cull_backfaces != 0)) {
      face_box(f, sqrt_blur, box.x, box.y, box.z, box.w);
      int ix_lo, ix_hi, iy_lo, iy_hi;
      exact_pixel_range(box.x, box.y, W, rx, ix_lo, ix_hi);
      exact_pixel_range(box.z, box.w, H, ry, iy_lo, iy_hi);
      if (ix_lo <= ix_hi && iy_lo <= iy_hi) {
        rng = make_int4(W - 1 - ix_hi, W - 1 - ix_lo, H - 1 - iy_hi, H - 1 - iy_lo);
        r = make_uint2((uint32_t)(rng.x / FTW) | ((uint32_t)(rng.y / FTW) << 16),
                       (uint32_t)(rng.z / FTH) | ((uint32_t)(rng.w / FTH) << 16));
      }
    }
    rect[fi] = make_uint4(r.x, r.y, (uint32_t)max(n, 0), 0u);
    // the reference reads the int64 neighbour index into an int (rasterize_meshes.cu:186)
    const int nb = neighbor ? (int)__ldg(neighbor + fi) : -1;
    float4* out = rec + fi * 4;
    out[0] = make_float4(f.x0, f.y0, f.x1, f.y1);
    out[1] = make_float4(f.x2, f.y2, bary_denominator(f), __int_as_float((int)fi));
    out[2] = make_float4(f.z0, f.z1, f.z2, __int_as_float(nb));
    out[3] = sqrt_blur > 0.0f ? box
                              : make_float4(__int_as_float(rng.x), __int_as_float(rng.y), __int_as_float(rng.z),
                                            __int_as_float(rng.w));
  }
  pdl_wait();  // the counters are zeroed by the kernel this one is chained to (see zero_ints_kernel)
  warp_count_rect(r, n, TY, TX, tile_count, tid & 31);  // all lanes participate
}

// ------------------------------------------------------------------------------------------------
// Per-(pixel, face) evaluation: the arithmetic of CheckPixelInsideFace (rasterize_meshes.cu:152-177).
// ------------------------------------------------------------------------------------------------
struct Hit {
  float z, dist, b0, b1, b2;
};

// An exact depth tie at the far end of some pixel's queue was seen: the tile's result may depend on the order in which
// the faces arrive (see fine_tile_body).  One flag per CTA at a fixed place in the fine kernels' dynamic shared memory
// (FineStage::tie), written on the (rare) event itself: watching costs no register.
__device__ __forceinline__ void flag_tie();

// `full` / `max_z`: the pixel's queue already holds K hits, the farthest at depth max_z.  The reference
// discards a further hit unless pz < q_max_z (rasterize_meshes.cu:226), so such a face is dropped right after
// its depth is known -- before the three point-segment distances, the expensive part when blur_radius > 0.
// WATCH: flag the tile when the depth EQUALS the queue's farthest one (the outcome then depends on arrival order).
template <bool WATCH>
__device__ __forceinline__ bool eval_pixel_face(float px, float py, const Face& f, float den, float blur_radius,
                                                bool persp, bool clip, bool full, float max_z, Hit& h) {
  const float e0 = edge_fn(px, py, f.x1, f.y1, f.x2, f.y2);
  const float e1 = edge_fn(px, py, f.x2, f.y2, f.x0, f.y0);
  const float e2 = edge_fn(px, py, f.x0, f.y0, f.x1, f.y1);
  float w0 = fdiv(e0, den), w1 = fdiv(e1, den), w2 = fdiv(e2, den);  // BarycentricCoordsForward
  if (persp) bary_persp(w0, w1, w2, f.z0, f.z1, f.z2);
  float c0 = w0, c1 = w1, c2 = w2;
  if (clip) bary_clip(c0, c1, c2);
  const float pz = ffma(f.z2, c2, ffma(f.z0, c0, fmul(f.z1, c1)));
  if (!(pz >= 0.0f)) return false;  // behind the image plane (:163)
  if (full && !(pz < max_z)) {
    if (WATCH && pz == max_z) flag_tie();
    return false;
  }
  const bool inside = w0 > 0.0f && w1 > 0.0f && w2 > 0.0f;
  if (!inside && !(blur_radius > 0.0f)) return false;  // dist >= 0 >= blur_radius always rejects (:175)
  const float dist = point_tri_dist(px, py, f);
  if (!inside && dist >= blur_radius) return false;
  h.z = pz;
  h.dist = inside ? -dist : dist;
  h.b0 = c0;
  h.b1 = c1;
  h.b2 = c2;
  return true;
}

__device__ __forceinline__ bool key_less(float za, int ia, float zb, int ib) {
  return za < zb || (za == zb && ia < ib);  // operator< of the reference's Pixel (rasterize_meshes.cu:30-32)
}

// The K nearest hits of one pixel.  This is the reference's per-pixel queue (rasterize_meshes.cu:179-237):
// an UNSORTED array of K slots plus the tracked maximum (q_max_z, q_max_idx); a new hit fills the next free
// slot, or -- when the queue is full and pz < q_max_z -- overwrites the tracked maximum, after which the
// maximum is searched again (first slot with a strictly larger z wins).  Faces reach the queue in ascending
// index order (sorted tile lists), so ties are resolved exactly as by the reference's naive kernel.
// The keys (z, face) live in registers with compile-time indices only (predicated updates); the payload
// (signed distance + barycentrics) of slot k lives in shared memory at pay[k * FTHREADS + thread], where
// a dynamic slot index costs nothing.
template <int KMAX>
struct TopK {
  float z[KMAX];
  int id[KMAX];
  int size;
  float max_z;
  int max_idx;

  __device__ __forceinline__ void init() {
#pragma unroll
    for (int i = 0; i < KMAX; ++i) {
      z[i] = -1.0f;
      id[i] = -1;
    }
    size = 0;
    max_z = -1000.0f;  // (:292)
    max_idx = -1;
  }
  __device__ __forceinline__ void put(int slot, const Hit& h, int f, float4* pay) {
#pragma unroll
    for (int i = 0; i < KMAX; ++i) {
      const bool w = i == slot;
      z[i] = w ? h.z : z[i];
      id[i] = w ? f : id[i];
    }
    pay[slot * FTHREADS] = make_float4(h.dist, h.b0, h.b1, h.b2);
  }
  // Handle a face that covers the pixel (the `else` branch at :216-236).
  __device__ __forceinline__ void offer(const Hit& h, int f, int K, float4* pay) {
    if (size < K) {
      put(size, h, f, pay);
      if (h.z > max_z) {
        max_z = h.z;
        max_idx = size;
      }
      ++size;
    } else if (h.z < max_z) {
      const float evicted = max_z;
      put(max_idx, h, f, pay);
      max_z = h.z;
#pragma unroll
      for (int i = 0; i < KMAX; ++i) {
        if (i < K && z[i] > max_z) {
          max_z = z[i];
          max_idx = i;
        }
      }
      if (max_z == evicted) flag_tie();  // another entry shares the evicted depth: which one left depends on the order
    } else if (h.z == max_z) {
      flag_tie();
    }
  }
  // Clipped-face neighbour handling (:186-215): if the other half of a clipped quad is already queued,
  // keep whichever half is closer to the pixel.  Returns true if the hit was consumed here.
  __device__ __forceinline__ bool offer_neighbor(const Hit& h, int f, int neighbor, float4* pay) {
    int at = -1;
#pragma unroll
    for (int i = KMAX - 1; i >= 0; --i)
      if (i < size && id[i] == neighbor) at = i;  // first match
    if (at < 0) return false;
    if (fabsf(h.dist) < fabsf(pay[at * FTHREADS].x)) {
      put(at, h, f, pay);
      if (h.z > max_z) {
        max_z = h.z;
        max_idx = at;
      }
    }
    return true;
  }
  // BubbleSort(q, q_size) on (z, idx) (:322 / rasterization_utils.cuh:52-66).  Keys are unique, so any
  // sorting network gives the same result; unfilled slots are pushed to the end.  slot[k] = queue slot (and
  // payload row) of the k-th nearest hit.
  __device__ __forceinline__ void sort(int (&slot)[KMAX]) {
    // only the first `n` slots (n = the largest queue of the warp, so that the branches below are uniform)
    // can hold hits: n rounds of odd-even transposition over those slots sort them.  Most pixels see a few
    // layers of surface, so this is typically one or zero compare-exchanges instead of KMAX^2 / 2.
    const int n = __reduce_max_sync(0xffffffffu, size);
#pragma unroll
    for (int i = 0; i < KMAX; ++i) {
      slot[i] = i;
      if (i >= size) {
        z[i] = FLT_MAX;
        id[i] = INT_MAX;
      }
    }
#pragma unroll
    for (int r = 0; r < KMAX; ++r) {
      if (r >= n) break;
#pragma unroll
      for (int i = r & 1; i + 1 < KMAX; i += 2) {
        if (i + 1 < n) {
          const bool sw = key_less(z[i + 1], id[i + 1], z[i], id[i]);
          const float za = z[i], zb = z[i + 1];
          z[i] = sw ? zb : za;
          z[i + 1] = sw ? za : zb;
          const int ia = id[i], ib = id[i + 1];
          id[i] = sw ? ib : ia;
          id[i + 1] = sw ? ia : ib;
          const int sa = slot[i], sb = slot[i + 1];
          slot[i] = sw ? sb : sa;
          slot[i + 1] = sw ? sa : sb;
        }
      }
    }
  }
};

// Queue policy of the K <= 8 kernel: TopK in registers + payload columns in shared memory.
template <int KMAX>
struct RegQueue {
  TopK<KMAX> q;
  float4* pay;  // this thread's payload column
  int K;
  __device__ __forceinline__ void reset() { q.init(); }
  __device__ __forceinline__ bool full() const { return q.size >= K; }
  __device__ __forceinline__ float max_z() const { return q.max_z; }
  __device__ __forceinline__ void offer(const Hit& h, int f) { q.offer(h, f, K, pay); }
  __device__ __forceinline__ bool offer_neighbor(const Hit& h, int f, int nb) { return q.offer_neighbor(h, f, nb, pay); }
};

// Queue policy of the 8 < K <= 32 kernel: the same queue with its keys in dynamic shared memory, slot-major with
// one column per thread (element k of this thread at [k * FTHREADS]) -- a dynamic slot index is free there, and
// a 32-slot queue in registers would cost 64 registers plus 2 * KMAX predicated moves per insertion.  Only
// (z, face) are kept (plus the signed distance when the clipped-face neighbour rule needs it); the barycentrics
// of the K winners are recomputed in the epilogue with the same arithmetic, hence the same bits.
template <bool NB>
struct SmemQueue {
  float* qz;
  int* qi;
  float* qd;  // NB only
  int K, size, max_idx;
  float max_zv;
  __device__ __forceinline__ void init(unsigned char* base, int K_, int tid) {
    K = K_;
    qz = reinterpret_cast<float*>(base) + tid;
    qi = reinterpret_cast<int*>(base) + K_ * FTHREADS + tid;
    qd = NB ? reinterpret_cast<float*>(base) + 2 * K_ * FTHREADS + tid : nullptr;
    reset();
  }
  __device__ __forceinline__ void reset() {
    size = 0;
    max_idx = -1;
    max_zv = -1000.0f;  // (:292)
  }
  __device__ __forceinline__ bool full() const { return size >= K; }
  __device__ __forceinline__ float max_z() const { return max_zv; }
  __device__ __forceinline__ void put(int slot, const Hit& h, int f) {
    qz[slot * FTHREADS] = h.z;
    qi[slot * FTHREADS] = f;
    if (NB) qd[slot * FTHREADS] = h.dist;
  }
  __device__ __forceinline__ void offer(const Hit& h, int f) {  // (:216-236)
    if (size < K) {
      put(size, h, f);
      if (h.z > max_zv) {
        max_zv = h.z;
        max_idx = size;
      }
      ++size;
    } else if (h.z < max_zv) {
      const float evicted = max_zv;
      put(max_idx, h, f);
      max_zv = h.z;
      for (int i = 0; i < K; ++i) {
        const float v = qz[i * FTHREADS];
        if (v > max_zv) {
          max_zv = v;
          max_idx = i;
        }
      }
      if (max_zv == evicted) flag_tie();
    } else if (h.z == max_zv) {
      flag_tie();
    }
  }
  __device__ __forceinline__ bool offer_neighbor(const Hit& h, int f, int nb) {  // (:186-215)
    int at = -1;
    for (int i = 0; i < size; ++i)
      if (qi[i * FTHREADS] == nb) {
        at = i;
        break;
      }
    if (at < 0) return false;
    if (NB && fabsf(h.dist) < fabsf(qd[at * FTHREADS])) {
      put(at, h, f);
      if (h.z > max_zv) {
        max_zv = h.z;
        max_idx = at;
      }
    }
    return true;
  }
  // BubbleSort on (z, idx) (:322): keys are unique -> an insertion sort over the thread's own column
  __device__ __forceinline__ void sort() {
    for (int i = 1; i < size; ++i) {
      const float tz = qz[i * FTHREADS];
      const int ti = qi[i * FTHREADS];
      int j = i - 1;
      while (j >= 0 && key_less(tz, ti, qz[j * FTHREADS], qi[j * FTHREADS])) {
        qz[(j + 1) * FTHREADS] = qz[j * FTHREADS];
        qi[(j + 1) * FTHREADS] = qi[j * FTHREADS];
        --j;
      }
      qz[(j + 1) * FTHREADS] = tz;
      qi[(j + 1) * FTHREADS] = ti;
    }
  }
};

// Shared-memory face records of one staged chunk of the large-K kernel (mesh_fine_bigk_kernel), which stages from
// face_verts itself; the K <= 32 kernels copy the setup pass's records instead (FineStage below).
struct __align__(16) FaceChunk {
  float4 box[CHUNK];  // xmin, xmax, ymin, ymax (blur-expanded; empty box = never hit)
  float4 a[CHUNK];    // x0, y0, x1, y1
  float4 b[CHUNK];    // x2, y2, den, face index (int bits)
  float4 c[CHUNK];    // z0, z1, z2, clipped-face neighbour index (int bits, -1 = none)
};

__device__ __forceinline__ void stage_face(FaceChunk& s, int slot, const float* __restrict__ face_verts,
                                           const int64_t* __restrict__ neighbor, int f, float sqrt_blur,
                                           bool cull_backfaces) {
  const float* v = face_verts + (int64_t)f * 9;
  const Face fc = {__ldg(v + 0), __ldg(v + 1), __ldg(v + 2), __ldg(v + 3), __ldg(v + 4),
                   __ldg(v + 5), __ldg(v + 6), __ldg(v + 7), __ldg(v + 8)};
  float xmin = FLT_MAX, xmax = -FLT_MAX, ymin = FLT_MAX, ymax = -FLT_MAX;
  if (face_is_drawable(fc, cull_backfaces)) face_box(fc, sqrt_blur, xmin, xmax, ymin, ymax);
  s.box[slot] = make_float4(xmin, xmax, ymin, ymax);
  s.a[slot] = make_float4(fc.x0, fc.y0, fc.x1, fc.y1);
  s.b[slot] = make_float4(fc.x2, fc.y2, bary_denominator(fc), __int_as_float(f));
  // the reference reads the int64 neighbour index into an int (:186)
  const int nb = neighbor ? (int)__ldg(neighbor + f) : -1;
  s.c[slot] = make_float4(fc.z0, fc.z1, fc.z2, __int_as_float(nb));
}

// Fragments are written once and read by a later kernel: streaming stores (evict-first) keep them from pushing
// the tile lists and face records, which the next tiles are about to read, out of L2.
template <typename T>
__device__ __forceinline__ void out_store(T* ptr, const T v) {
  __stcs(ptr, v);
}

struct FineParams {
  const float* face_verts;
  const int64_t* neighbor;  // clipped_faces_neighbor_idx or nullptr
  const float4* rec;
  const int64_t* first;
  const int64_t* num;
  const int* tile_offset;
  const int* tile_order;  // schedule: the CTA with linear index b takes tile tile_order[b] (nullptr: tile b)
  int* pairs;  // tile lists; each CTA puts its own segment in ascending face order before reading it
  int64_t capacity;
  int n0;  // first image of this launch (grid.z is limited to 65535 images)
  int N, H, W, K, TY, TX;
  float rx, ry, blur_radius, sqrt_blur;
  int persp, clip, cull;
  int smem_ints;  // dynamic shared memory of the launch, in 4-byte words (scratch of the in-kernel list sort)
  int64_t* pix_to_face;
  float* zbuf;
  float* bary;
  float* dists;
};

// Pixel owned by this thread: warp w covers an 8 (x) by 4 (y) footprint of the 16x16 tile.
__device__ __forceinline__ void thread_pixel(int tile_x, int tile_y, int& xo, int& yo) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  xo = tile_x * TILE + (w & 1) * 8 + (lane & 7);
  yo = tile_y * TILE + (w >> 1) * 4 + (lane >> 3);
}
// ... of the forward pass's FTW x FTH tiles
__device__ __forceinline__ void fthread_pixel(int tile_x, int tile_y, int& xo, int& yo) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  xo = tile_x * FTW + (w & 1) * 8 + (lane & 7);
  yo = tile_y * FTH + (w >> 1) * 4 + (lane >> 3);
}

__device__ __forceinline__ float warp_min(float v) {
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) v = fminf(v, __shfl_xor_sync(0xffffffffu, v, d));
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, d));
  return v;
}

// Blur > 0: faces are consumed in rounds of 64.  Pass A: each lane box-tests one face against the whole footprint
// and the warp transposes the resulting bit matrix, so that every lane ends up with a 64-bit mask of the faces
// whose box contains ITS pixel (ascending face order = ascending bit order).  Pass B: every lane walks its
// own mask.  In pass A the warp does ~80 instructions per 32 faces no matter how many survive; in pass B
// each lane works on a different face that is known to touch its pixel, so the expensive arithmetic runs on
// (nearly) full warps even when triangles are pixel-sized and only a handful of the footprint's 32 pixels
// lie in a given face's box.
constexpr int ROUND = 64;

// Staging area of the fine kernels (21 KB), at the start of their dynamic shared memory; the queue storage follows.
struct FineStage {
  float4 a[CHUNK];  // x0, y0, x1, y1            } the staged chunk: copies of the per-face records
  float4 b[CHUNK];  // x2, y2, den, face index   }
  float4 c[CHUNK];  // z0, z1, z2, neighbour     }
  union {
    float4 box[CHUNK];                          // blur > 0: blur-expanded boxes (pass A)
    unsigned mask[CHUNK / 32][FTHREADS];        // blur = 0: per pixel (thread), one bit per staged face
    int sort_buf[2 * FTHREADS];                 // exchange buffers of cta_sort256 (before the chunk is staged)
  } u;
  unsigned rng[CHUNK];                          // blur = 0: tile-local pixel rectangle c_lo | c_hi<<8 | r_lo<<16 | r_hi<<24
  float col[FTW], row[FTH];                     // NDC coordinates of the tile's pixel columns / rows
  int tie;                                      // see flag_tie()
};

__device__ __forceinline__ void flag_tie() {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  reinterpret_cast<FineStage*>(smem_raw)->tie = 1;
}

// Full-sector output stores.  A pixel's K values of one buffer are P 16-byte pieces; the pixels of two adjacent
// lanes (x, x+1 of the same row) are adjacent in memory, a run of 2P pieces.  Written lane-by-lane, every store
// instruction would fill only half of each 32-byte sector it touches (the other half comes with a later
// instruction): twice the L1->L2 write transactions.  Instead the two lanes exchange half of their pieces with
// one shuffle round per two pieces, so that in instruction j the even lane writes piece 2j and the odd lane
// piece 2j+1 of the run -- whole sectors.  `mine` = this lane's P pieces; `run` = start of the pair's run;
// vA / vB = whether the even / odd lane's pixel exists (partial tiles).
template <int P>
__device__ __forceinline__ void store_pair_run(float4* run, const float4 (&mine)[P], int odd, bool vA, bool vB) {
  constexpr int H = P / 2;           // pieces received from the partner
  constexpr int CE = (P + 1) / 2;    // first instruction whose even-lane piece belongs to the odd lane's pixel
  float4 recv[H > 0 ? H : 1];
#pragma unroll
  for (int r = 0; r < H; ++r) {
    // the odd lane needs A[2r+1]; the even lane needs B[2 * (CE + r) - P]
    const float4 send = odd ? mine[2 * (CE + r) - P] : mine[2 * r + 1];
    recv[r].x = __shfl_xor_sync(0xffffffffu, send.x, 1);
    recv[r].y = __shfl_xor_sync(0xffffffffu, send.y, 1);
    recv[r].z = __shfl_xor_sync(0xffffffffu, send.z, 1);
    recv[r].w = __shfl_xor_sync(0xffffffffu, send.w, 1);
  }
#pragma unroll
  for (int j = 0; j < P; ++j) {
    // even lane: run piece 2j (its own while 2j < P); odd lane: run piece 2j+1 (its own once 2j+1 >= P)
    const float4 ve = 2 * j < P ? mine[2 * j < P ? 2 * j : 0] : recv[j >= CE ? j - CE : 0];
    const float4 vo = 2 * j + 1 < P ? recv[2 * j + 1 < P ? j : 0] : mine[2 * j + 1 >= P ? 2 * j + 1 - P : 0];
    const bool target_a = odd ? (2 * j + 1 < P) : (2 * j < P);
    if (target_a ? vA : vB) out_store(run + 2 * j + odd, odd ? vo : ve);
  }
}

// The same for two separate runs of P (even) pieces each: `runA` belongs to the even lane's pixel, `runB` to the
// odd lane's (a group of 8 slots of a pixel with K > 8: the two pixels' groups are K slots apart).  The lanes
// swap every other piece, then both write run A (even lane piece 2r, odd lane piece 2r+1: one whole sector per
// pair and instruction), then run B.
template <int P>
__device__ __forceinline__ void store_pair_split(float4* runA, float4* runB, const float4 (&mine)[P], int odd,
                                                 bool vA, bool vB) {
  static_assert(P % 2 == 0, "an even number of 16-byte pieces per run");
  float4 recv[P / 2];  // even lane: B[2r]; odd lane: A[2r+1]
#pragma unroll
  for (int r = 0; r < P / 2; ++r) {
    const float4 send = odd ? mine[2 * r] : mine[2 * r + 1];
    recv[r].x = __shfl_xor_sync(0xffffffffu, send.x, 1);
    recv[r].y = __shfl_xor_sync(0xffffffffu, send.y, 1);
    recv[r].z = __shfl_xor_sync(0xffffffffu, send.z, 1);
    recv[r].w = __shfl_xor_sync(0xffffffffu, send.w, 1);
  }
#pragma unroll
  for (int r = 0; r < P / 2; ++r)
    if (vA) out_store(runA + 2 * r + odd, odd ? recv[r] : mine[2 * r]);
#pragma unroll
  for (int r = 0; r < P / 2; ++r)
    if (vB) out_store(runB + 2 * r + odd, odd ? mine[2 * r + 1] : recv[r]);
}

// A tile no face touches: all of its outputs are -1.  Full tiles are written as whole 16-pixel row segments
// (consecutive lanes -> consecutive 16 bytes) without computing anything per pixel.  KMAX > 0: K == KMAX is
// checked and the loops are unrolled; KMAX == 0: any K that is a multiple of 4.
template <int KMAX>
__device__ __forceinline__ void write_empty_tile(const FineParams& p, int n, int tile_x, int tile_y) {
  const int tid = threadIdx.x;
  const int x0 = tile_x * FTW, y0 = tile_y * FTH;
  const int K = p.K;
  if ((KMAX == 0 || K == KMAX) && (K % 4) == 0 && x0 + FTW <= p.W && y0 + FTH <= p.H) {
    const float4 m1 = make_float4(-1.f, -1.f, -1.f, -1.f);
    const int KK = KMAX > 0 ? KMAX : K;
    const int SEG_I = FTW * KK / 2;  // longlong2 per row segment of pix_to_face
    const int SEG_F = FTW * KK / 4;  // float4 per row segment of zbuf / dists (x3 for bary)
#pragma unroll
    for (int e = tid; e < FTH * SEG_I; e += FTHREADS) {
      const int64_t o = (((int64_t)n * p.H + y0 + e / SEG_I) * p.W + x0) * KK;
      out_store(reinterpret_cast<longlong2*>(p.pix_to_face + o) + e % SEG_I, make_longlong2(-1ll, -1ll));
    }
#pragma unroll
    for (int e = tid; e < FTH * SEG_F; e += FTHREADS) {
      const int64_t o = (((int64_t)n * p.H + y0 + e / SEG_F) * p.W + x0) * KK;
      out_store(reinterpret_cast<float4*>(p.zbuf + o) + e % SEG_F, m1);
      out_store(reinterpret_cast<float4*>(p.dists + o) + e % SEG_F, m1);
    }
#pragma unroll
    for (int e = tid; e < FTH * SEG_F * 3; e += FTHREADS) {
      const int64_t o = (((int64_t)n * p.H + y0 + e / (SEG_F * 3)) * p.W + x0) * KK;
      out_store(reinterpret_cast<float4*>(p.bary + o * 3) + e % (SEG_F * 3), m1);
    }
    return;
  }
  int xo, yo;
  fthread_pixel(tile_x, tile_y, xo, yo);
  if (xo >= p.W || yo >= p.H) return;
  const int64_t o = (((int64_t)n * p.H + yo) * p.W + xo) * K;
  for (int k = 0; k < K; ++k) {
    p.pix_to_face[o + k] = -1ll;
    p.zbuf[o + k] = -1.0f;
    p.dists[o + k] = -1.0f;
    p.bary[(o + k) * 3 + 0] = -1.0f;
    p.bary[(o + k) * 3 + 1] = -1.0f;
    p.bary[(o + k) * 3 + 2] = -1.0f;
  }
}

// One candidate face (staged at slot j) against this thread's pixel.
template <class Q, bool NB>
__device__ __forceinline__ void consider_face(const FineStage& sh, int j, float px, float py, float blur_radius,
                                              bool persp, bool clip, Q& q) {
  const float4 fa = sh.a[j], fb = sh.b[j], fc = sh.c[j];
  const Face f = {fa.x, fa.y, fc.x, fa.z, fa.w, fc.y, fb.x, fb.y, fc.z};
  const int nb = NB ? __float_as_int(fc.w) : -1;
  Hit h;
  // (a face with a clipped-face neighbour may replace that neighbour whatever its depth: no early rejection)
  if (!eval_pixel_face<true>(px, py, f, fb.z, blur_radius, persp, clip, q.full() && nb == -1, q.max_z(), h)) return;
  const int fi = __float_as_int(fb.w);
  if (NB && nb != -1 && q.offer_neighbor(h, fi, nb)) return;
  q.offer(h, fi);
}

// Depth culling for a whole warp (blur > 0: every face in the blur band of a pixel is a hit, tens to thousands per pixel,
// of which only the K nearest survive).  Once every pixel of the warp's footprint holds K hits, a face can only matter if
// its depth at some pixel of the footprint is below `zcut`, the largest of those pixels' farthest kept depths -- the
// queue itself discards a hit unless pz < max_z (rasterize_meshes.cu:226).  face_depth_lower_bound returns a rigorous lower
// bound of the depth the kernel would COMPUTE for any pixel of the footprint (so dropping the face cannot change any
// result, whatever the order of the walk), or -FLT_MAX when no bound is available:
//   clip_barycentric_coords: the clipped, renormalised barycentrics are a convex combination (each in [0, 1], sum within
//     3 ulp of 1), and drawable faces have zmin >= 1e-8 > 0: pz >= zmin * (1 - 1e-6).
//   neither clip nor perspective correction: pz is, in exact arithmetic, the affine function
//     (z0 E0(p) + z1 E1(p) + z2 E2(p)) / den of the pixel; its minimum over the footprint's rectangle is the value at the
//     centre minus |gradient| . half-extent; the float evaluation of any pixel differs from the exact value by at most
//     27 ulp-units of zabs * M / |den| (M bounds every product inside the edge functions over the footprint) -- the
//     margin below takes 1e-5 (> 160 * 2^-24) of that plus 1e-5 of the bound's own terms.
//   perspective correction without clipping: no bound (the face is kept).
__device__ __forceinline__ float face_depth_lower_bound(const float4 fa, const float4 fb, const float4 fc, float cx,
                                                        float cy, float hx, float hy, bool persp, bool clip) {
  const float z0 = fc.x, z1 = fc.y, z2 = fc.z;
  if (clip) return fminf(fminf(z0, z1), z2) * (1.0f - 1e-6f);
  if (persp) return -FLT_MAX;
  const float x0 = fa.x, y0 = fa.y, x1 = fa.z, y1 = fa.w, x2 = fb.x, y2 = fb.y;
  const float rd = 1.0f / fabsf(fb.z);
  const float e0 = (cx - x1) * (y2 - y1) - (cy - y1) * (x2 - x1);
  const float e1 = (cx - x2) * (y0 - y2) - (cy - y2) * (x0 - x2);
  const float e2 = (cx - x0) * (y1 - y0) - (cy - y0) * (x1 - x0);
  const float num = z0 * e0 + z1 * e1 + z2 * e2;
  const float gxn = z0 * (y2 - y1) + z1 * (y0 - y2) + z2 * (y1 - y0);
  const float gyn = z0 * (x2 - x1) + z1 * (x0 - x2) + z2 * (x1 - x0);
  const float pzc = (fb.z < 0.0f ? -num : num) * rd;
  const float spread = (fabsf(gxn) * hx + fabsf(gyn) * hy) * rd;
  const float dx = fmaxf(fmaxf(fabsf(cx - x0), fabsf(cx - x1)), fabsf(cx - x2)) + hx;
  const float dy = fmaxf(fmaxf(fabsf(cy - y0), fabsf(cy - y1)), fabsf(cy - y2)) + hy;
  const float lx = fmaxf(fmaxf(x0, x1), x2) - fminf(fminf(x0, x1), x2);
  const float ly = fmaxf(fmaxf(y0, y1), y2) - fminf(fminf(y0, y1), y2);
  const float zabs = fmaxf(fmaxf(fabsf(z0), fabsf(z1)), fabsf(z2));
  const float margin = 1e-5f * (zabs * (dx * ly + dy * lx) * rd + fabsf(pzc) + spread);
  const float lb = pzc - spread - margin;
  return lb == lb ? lb : -FLT_MAX;  // (NaN / inf coordinates: no bound)
}

// The body shared by the fine kernels: stage the tile's list chunk by chunk, find every pixel's candidates and offer
// the hits to the pixel's queue `q`.
//
// Order of the list.  The fill pass scatters with atomics, so a tile's list arrives in arbitrary order, while the
// reference's naive kernel offers faces in ascending index order (rasterize_meshes.cu:301).  Its queue keeps the K
// nearest hits whatever the order UNLESS two hits share, bit for bit, the depth at the queue's far end (a full queue
// meets a hit with z == q_max_z, or evicts one of several entries at q_max_z); the final sort on (z, face) is
// order-free.  So without a blur band -- where such ties are rare: none on the north-star batch -- the tile is first
// walked in arrival order with the queues watching for exactly those events (flag_tie()); only if some pixel saw one
// is the list sorted and the tile walked -- and written -- again (the kernels loop: walk, epilogue, tile_saw_tie()).  With a blur band (structured meshes tie often there: the two
// triangles of a quad extrapolate to the same depth) and with clipped-face neighbours (whose replace-in-queue rule
// depends on the order by itself) the list is sorted up front.  Either way the result is the one the sorted walk
// gives; sorting every list cost 30 % of the kernel's instructions.
// `order`: ORDER_ARRIVAL (the list as the fill pass left it) or ORDER_INDEX (ascending face index: the reference's
// order).  `valid`: this thread's pixel lies in the image (its queue is updated); the others still help to stage.
enum { ORDER_ARRIVAL = 0, ORDER_INDEX = 1 };

template <class Q, bool NB, bool SCAN>
__device__ __forceinline__ void fine_tile_body(const FineParams& p, FineStage& sh, Q& q, int tile_x, int tile_y, int n,
                                               int seg_begin, int count, bool overflow, int order, bool valid, int lc,
                                               int lr) {
  const int tid = threadIdx.x, lane = tid & 31;
  const bool persp = p.persp != 0, clip = p.clip != 0;
  const float blur_radius = p.blur_radius;
  // (an overflowed tile walks the mesh's own faces: already in order)
  const bool sorted_walk = order == ORDER_INDEX;
  const bool sort_staged = sorted_walk && !overflow && count <= CHUNK;
  // (the long-list sort uses the kernel's shared memory as scratch: nothing lives there yet / any more)
  if (sorted_walk && !overflow && count > CHUNK)
    cta_sort_segment<FTHREADS>(p.pairs + seg_begin, count, reinterpret_cast<int*>(&sh), p.smem_ints);
  // NDC coordinates of the tile's 16 pixel columns and rows (two IEEE divisions each): computed once per tile
  // by 32 threads, read by every thread after the barriers of the first chunk
  if (tid < FTW + FTH) {
    if (tid < FTW)
      sh.col[tid] = pix_to_ndc(p.W - 1 - (tile_x * FTW + tid), p.W, p.rx);
    else
      sh.row[tid - FTW] = pix_to_ndc(p.H - 1 - (tile_y * FTH + tid - FTW), p.H, p.ry);
  }
  if (!sorted_walk && tid == FTW + FTH) sh.tie = 0;

  for (int base = 0; base < count; base += CHUNK) {
    const int nc = min(CHUNK, count - base);
    const int nwords = (nc + 31) >> 5;
    if (base > 0) __syncthreads();  // previous chunk fully consumed
    int f = INT_MAX;
    if (tid < nc) f = overflow ? (int)(p.first[n] + base + tid) : p.pairs[seg_begin + base + tid];
    if (sort_staged) {
      f = cta_sort256<FTHREADS>(f, nc, sh.u.sort_buf);
      if (nc > 32) __syncthreads();  // the exchange buffers alias the masks / boxes written next
    }
    if (tid < nc) {
      const float4* r = p.rec + (int64_t)f * 4;
      const float4 ra = __ldg(r + 0), rb = __ldg(r + 1), rc = __ldg(r + 2), rd = __ldg(r + 3);
      sh.a[tid] = ra;
      sh.b[tid] = rb;
      sh.c[tid] = rc;
      if (SCAN) {
        const int gx = __float_as_int(rd.x), gy = __float_as_int(rd.y), gz = __float_as_int(rd.z),
                  gw = __float_as_int(rd.w);
        const int c_lo = max(gx - tile_x * FTW, 0), c_hi = min(gy - tile_x * FTW, FTW - 1);
        const int r_lo = max(gz - tile_y * FTH, 0), r_hi = min(gw - tile_y * FTH, FTH - 1);
        sh.rng[tid] = (c_lo > c_hi || r_lo > r_hi) ? 1u  // empty: c_lo = 1 > c_hi = 0
                                                   : (unsigned)(c_lo | (c_hi << 8) | (r_lo << 16) | (r_hi << 24));
      } else {
        sh.u.box[tid] = rd;
      }
    }
    if (SCAN) {
      for (int w = 0; w < nwords; ++w) sh.u.mask[w][tid] = 0u;
    }
    __syncthreads();
    if (SCAN) {
      // ---- scan conversion (no blur band): a hit requires the pixel to be strictly inside the face, i.e. all
      //      three w_i = E_i / den > 0, which implies that every edge function E_i is non-zero and has the sign
      //      of den -- a test that needs no division.  Four lanes take one face and walk the rows of its pixel
      //      rectangle (exactly the set of pixels that pass the reference's box test; precomputed per face by
      //      the setup pass, here clamped to the tile); a pixel that passes gets the face's bit set in its mask.
      //      The search costs ~(pixels in the box) per face instead of ~(faces in the tile) per pixel, and
      //      leaves the candidates of every pixel in ascending face order.  (Measured on the NS workload:
      //      1x2 / 1x4 lanes per face 186 us, 2x2 200 us, 4x4 215 us, 8x2 270 us -- the loop-invariant part of a
      //      face is amortised over more pixels with fewer lanes.)
      constexpr int SL = 4;  // lanes per face (also timed: 1, 2)
      const int dr = tid & (SL - 1);
      for (int fslot = tid / SL; fslot < nc; fslot += FTHREADS / SL) {
        const unsigned rg = sh.rng[fslot];
        const int c_lo = rg & 255, c_hi = (rg >> 8) & 255, r_lo = (rg >> 16) & 255, r_hi = rg >> 24;
        if (c_lo > c_hi) continue;
        const float4 fa = sh.a[fslot], fb = sh.b[fslot];
        const bool pos = fb.z > 0.0f;
        unsigned* mrow = sh.u.mask[fslot >> 5];
        const unsigned bit = 1u << (fslot & 31);
        // edge_fn(q; a, b) = fma(q.x - a.x, b.y - a.y, -rn((q.y - a.y) * (b.x - a.x))): the differences of the
        // face's own vertices are per-face constants, the rounded product is a per-row constant
        const float dx0 = fsub(fb.x, fa.z), dy0 = fsub(fb.y, fa.w);  // v2 - v1
        const float dx1 = fsub(fa.x, fb.x), dy1 = fsub(fa.y, fb.y);  // v0 - v2
        const float dx2 = fsub(fa.z, fa.x), dy2 = fsub(fa.w, fa.y);  // v1 - v0
        for (int r = r_lo + dr; r <= r_hi; r += SL) {
          const float qy = sh.row[r];
          const float t0 = fmul(fsub(qy, fa.w), dx0), t1 = fmul(fsub(qy, fb.y), dx1), t2 = fmul(fsub(qy, fa.y), dx2);
          unsigned* mpix = mrow + (r >> 2) * 64 + (r & 3) * 8;  // thread of pixel (r, c): + (c / 8) * 32 + c % 8
          for (int c0 = c_lo; c0 <= c_hi; c0 += 4) {
#pragma unroll
            for (int u = 0; u < 4; ++u) {  // four columns in flight
              const int c = c0 + u;
              if (c <= c_hi) {
                const float qx = sh.col[c];
                const float e0 = ffma(fsub(qx, fa.z), dy0, -t0);  // E(p; v1, v2)
                const float e1 = ffma(fsub(qx, fb.x), dy1, -t1);  // E(p; v2, v0)
                const float e2 = ffma(fsub(qx, fa.x), dy2, -t2);  // E(p; v0, v1)
                const bool ok = pos ? (e0 > 0.0f && e1 > 0.0f && e2 > 0.0f) : (e0 < 0.0f && e1 < 0.0f && e2 < 0.0f);
                if (ok) atomicOr(mpix + (c >> 3) * 32 + (c & 7), bit);
              }
            }
          }
        }
      }
      __syncthreads();
      // every pixel walks its own candidates, in ascending face order.  A pixel has a handful of candidates spread
      // over the chunk's mask words; every lane advances through ITS words on its own (skipping empty ones costs three
      // instructions), so that the lanes of a warp evaluate their n-th candidates together whatever words those are
      // in -- looping over the words in lockstep left a third of the lanes active in the evaluation (ncu: 9.8 of 32).
      const float px = sh.col[lc], py = sh.row[lr];
      {
        int w = 0;
        unsigned m = sh.u.mask[0][tid];
        for (;;) {
          while (m == 0u && ++w < nwords) m = sh.u.mask[w][tid];
          if (m == 0u) break;
          const int j = w * 32 + __ffs((int)m) - 1;
          m &= m - 1u;
          consider_face<Q, NB>(sh, j, px, py, blur_radius, persp, clip, q);
        }
      }
      continue;  // chunk done
    }
    const float px = sh.col[lc], py = sh.row[lr];
    // (worth its ~80 instructions per face and warp only where a pixel has far more candidates than queue slots: long
    // tile lists -- config 5: 2300 faces per tile, 13.0 -> 9.1 ms; north-star batch with blur 1e-4: none culled, +3 %)
    const bool cull_depth = (clip || !persp) && count >= 512;
    // extent of the warp's footprint (pixel centres are monotonic in the pixel index)
    const float fc0 = sh.col[lc & 8], fc1 = sh.col[(lc & 8) + 7], fr0 = sh.row[lr & 12], fr1 = sh.row[(lr & 12) + 3];
    const float cmin = fminf(fc0, fc1), cmax = fmaxf(fc0, fc1), rmin = fminf(fr0, fr1), rmax = fmaxf(fr0, fr1);
    const bool warp_active = __any_sync(0xffffffffu, valid);  // (false for a warp wholly outside the image)
    for (int sub = 0; sub < nc; sub += ROUND) {
      if (!warp_active) break;
      // ---- pass A: 64-bit mask of the faces of this round whose box contains my pixel
      unsigned m0 = 0, m1 = 0;
      {
        // A blur band wider than the footprint (32 px boxes at blur_radius 1e-3 on 1024^2) makes most boxes contain the
        // WHOLE footprint: when that holds for all 32 faces of a half-round the bit matrix is all ones -- four
        // compares and a vote instead of twelve compares, the bit assembly and five shuffle stages.
        const bool h0 = sub + lane < nc, h1 = sub + 32 + lane < nc;
        float4 b0 = make_float4(FLT_MAX, -FLT_MAX, FLT_MAX, -FLT_MAX), b1 = b0;
        if (h0) b0 = sh.u.box[sub + lane];
        if (h1) b1 = sh.u.box[sub + 32 + lane];
        // depth culling (see face_depth_lower_bound): once every pixel of the footprint holds K hits
        bool keep0 = h0, keep1 = h1;
        if (cull_depth) {
          const float zcut = warp_max(!valid ? -FLT_MAX : (q.full() ? q.max_z() : FLT_MAX));
          if (zcut < FLT_MAX) {
            const float cx = 0.5f * (cmin + cmax), cy = 0.5f * (rmin + rmax);
            const float hx = 0.5f * (cmax - cmin) * (1.0f + 1e-6f), hy = 0.5f * (rmax - rmin) * (1.0f + 1e-6f);
            if (h0) {
              const float4 fc = sh.c[sub + lane];
              if (!NB || __float_as_int(fc.w) == -1)
                keep0 = !(face_depth_lower_bound(sh.a[sub + lane], sh.b[sub + lane], fc, cx, cy, hx, hy, persp, clip) >
                          zcut);
            }
            if (h1) {
              const float4 fc = sh.c[sub + 32 + lane];
              if (!NB || __float_as_int(fc.w) == -1)
                keep1 = !(face_depth_lower_bound(sh.a[sub + 32 + lane], sh.b[sub + 32 + lane], fc, cx, cy, hx, hy,
                                                 persp, clip) > zcut);
            }
            if (!keep0) b0 = make_float4(FLT_MAX, -FLT_MAX, FLT_MAX, -FLT_MAX);
            if (!keep1) b1 = make_float4(FLT_MAX, -FLT_MAX, FLT_MAX, -FLT_MAX);
            if (!__any_sync(0xffffffffu, keep0 || keep1)) continue;  // the whole round lies behind the footprint
          }
        }
        // (every face of the half-round is either absent / culled or contains the whole footprint)
        const bool all0 =
            __all_sync(0xffffffffu, !keep0 || (cmin >= b0.x && cmax <= b0.y && rmin >= b0.z && rmax <= b0.w));
        const bool all1 =
            __all_sync(0xffffffffu, !keep1 || (cmin >= b1.x && cmax <= b1.y && rmin >= b1.z && rmax <= b1.w));
        if (all0 && all1) {
          m0 = __ballot_sync(0xffffffffu, keep0);
          m1 = __ballot_sync(0xffffffffu, keep1);
        } else {
          // the footprint's 8 column and 4 row coordinates (lane = row * 8 + column); re-gathered per round so
          // that they do not occupy 12 registers during pass B and the epilogue
          float col[8], row[4];
#pragma unroll
          for (int c = 0; c < 8; ++c) col[c] = sh.col[(lc & 8) + c];
#pragma unroll
          for (int r = 0; r < 4; ++r) row[r] = sh.row[(lr & 12) + r];
          if (keep0) m0 = box_pixel_mask(b0, col, row);
          if (keep1) m1 = box_pixel_mask(b1, col, row);
          m0 = warp_transpose_bits(m0, lane);
          if (sub + 32 < nc) m1 = warp_transpose_bits(m1, lane);
        }
      }
      unsigned long long mine = valid ? (((unsigned long long)m1 << 32) | m0) : 0ull;
      // ---- pass B: every lane evaluates its own candidates, in ascending face order
      while (__any_sync(0xffffffffu, mine != 0ull)) {
        if (mine != 0ull) {
          const int j = sub + __ffsll((long long)mine) - 1;
          mine &= mine - 1ull;
          consider_face<Q, NB>(sh, j, px, py, blur_radius, persp, clip, q);
        }
      }
    }
  }
}

// After the epilogue of an arrival-order walk: did any pixel of the tile see a depth tie?  CTA-uniform: every thread
// contributes its own view of the flag (the thread that raised it sees it) and nobody reads it after the barrier, which
// also orders every warp's epilogue reads of the queue payload before the sorted walk reuses shared memory.
__device__ __forceinline__ bool tile_saw_tie(const FineStage& sh) {
  return __syncthreads_or(sh.tie) != 0;
}

// Which tile, which faces: grid = (tiles per row, tile rows, images) -- no integer divisions.
struct TileWork {
  int tile_x, tile_y, n, seg_begin, count;
  bool overflow;
};
__device__ __forceinline__ TileWork tile_work(const FineParams& p) {
  pdl_wait();  // the tile lists (fill kernel) and, transitively, the face records are complete (see common.cuh)
  TileWork t;
  int i = ((p.n0 + blockIdx.z) * p.TY + blockIdx.y) * p.TX + blockIdx.x;  // linear index of this CTA
  if (p.tile_order != nullptr) {
    i = p.tile_order[i];  // heavy tiles first, empty tiles last (see tile_scan_kernel)
    t.tile_x = i % p.TX;
    const int r = i / p.TX;
    t.tile_y = r % p.TY;
    t.n = r / p.TY;
  } else {
    t.tile_x = blockIdx.x;
    t.tile_y = blockIdx.y;
    t.n = p.n0 + blockIdx.z;
  }
  // the tile's face list; tiles whose segment did not fit the pair buffer test every face of the mesh
  t.seg_begin = p.tile_offset[i];
  const int seg_end = p.tile_offset[i + 1];
  t.overflow = (int64_t)seg_end > p.capacity || seg_end == INT_MAX;
  t.count = t.overflow ? (int)p.num[t.n] : seg_end - t.seg_begin;
  return t;
}

// Which walk a tile starts with (see fine_tile_body and DESIGN.md 5): index order for overflowed tiles, for clipped-face
// neighbours (order-dependent by themselves) and with a blur band; otherwise arrival order, watched for depth ties.
// (A front-to-back walk of the blur band, with the pixels that saw a tie redone in index order, was measured slower:
// structured meshes tie so often in the band that too many pixels are redone -- north-star batch with blur 1e-4: fine
// 917 -> 1306 us, config 2: 139 -> 198 us, config 5: 9.3 -> 14.9 ms.)
template <bool NB, bool SCAN>
__device__ __forceinline__ int first_walk_order(const TileWork& t) {
  return (t.overflow || NB || !SCAN) ? ORDER_INDEX : ORDER_ARRIVAL;
}

template <int KMAX, bool NB, bool SCAN>
__global__ void __launch_bounds__(FTHREADS, 1024 / FTHREADS) mesh_fine_kernel(const FineParams p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  FineStage& sh = *reinterpret_cast<FineStage*>(smem_raw);
  const int tid = threadIdx.x, lane = tid & 31;
  const TileWork t = tile_work(p);
  const int tile_x = t.tile_x, tile_y = t.tile_y, n = t.n;
  if (t.count == 0) {
    write_empty_tile<KMAX>(p, n, tile_x, tile_y);
    return;
  }
  int xo, yo;
  fthread_pixel(tile_x, tile_y, xo, yo);
  const bool valid = xo < p.W && yo < p.H;
  const int lc = xo - tile_x * FTW, lr = yo - tile_y * FTH;  // local column / row of my pixel

  RegQueue<KMAX> rq;
  rq.q.init();
  rq.pay = reinterpret_cast<float4*>(smem_raw + sizeof(FineStage)) + tid;
  rq.K = p.K;
  TopK<KMAX>& q = rq.q;
  float4* pay = rq.pay;
  const int K = p.K;
  // (see fine_tile_body: arrival-order walk first where ties are rare, sorted walk only if one was seen)
  int order = first_walk_order<NB, SCAN>(t);
  for (;;) {
  fine_tile_body<RegQueue<KMAX>, NB, SCAN>(p, sh, rq, tile_x, tile_y, n, t.seg_begin, t.count, t.overflow, order,
                                           valid, lc, lr);
  bool stored = false;
  int slot[KMAX];
  q.sort(slot);
  // ---- epilogue: every output is written with 16-byte stores (all K slots, including the -1 padding)
  const int64_t o = (((int64_t)n * p.H + yo) * p.W + xo) * K;
  if constexpr ((KMAX % 4) == 0) {
   if (K == KMAX) {
    // lanes 2m / 2m+1 own horizontally adjacent pixels: they write their two pixels' runs together
    const int odd = lane & 1;
    const bool vA = __shfl_sync(0xffffffffu, (int)valid, lane & ~1) != 0;
    const bool vB = __shfl_sync(0xffffffffu, (int)valid, lane | 1) != 0;
    const int64_t oa = o - (int64_t)odd * KMAX;  // the even lane's pixel
    {
      // pix_to_face: int64, but the values are the queue's int32 face ids: exchange those, widen at the store
      float4 piece[KMAX / 2];
#pragma unroll
      for (int k = 0; k < KMAX; k += 2) {
        const long long i0 = k >= q.size ? -1ll : (long long)q.id[k];
        const long long i1 = k + 1 >= q.size ? -1ll : (long long)q.id[k + 1];
        piece[k / 2] = make_float4(__int_as_float((int)(i0 & 0xffffffffll)), __int_as_float((int)(i0 >> 32)),
                                   __int_as_float((int)(i1 & 0xffffffffll)), __int_as_float((int)(i1 >> 32)));
      }
      store_pair_run<KMAX / 2>(reinterpret_cast<float4*>(p.pix_to_face + oa), piece, odd, vA, vB);
    }
    {
      float4 piece[KMAX / 4];
#pragma unroll
      for (int k0 = 0; k0 < KMAX; k0 += 4)
        piece[k0 / 4] = make_float4(k0 + 0 >= q.size ? -1.0f : q.z[k0 + 0], k0 + 1 >= q.size ? -1.0f : q.z[k0 + 1],
                                    k0 + 2 >= q.size ? -1.0f : q.z[k0 + 2], k0 + 3 >= q.size ? -1.0f : q.z[k0 + 3]);
      store_pair_run<KMAX / 4>(reinterpret_cast<float4*>(p.zbuf + oa), piece, odd, vA, vB);
    }
    {
      float4 piece[KMAX / 4];
#pragma unroll
      for (int k0 = 0; k0 < KMAX; k0 += 4) {
        float d[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) d[u] = k0 + u >= q.size ? -1.0f : pay[slot[k0 + u] * FTHREADS].x;
        piece[k0 / 4] = make_float4(d[0], d[1], d[2], d[3]);
      }
      store_pair_run<KMAX / 4>(reinterpret_cast<float4*>(p.dists + oa), piece, odd, vA, vB);
    }
    {
      float4 piece[3 * KMAX / 4];
#pragma unroll
      for (int k0 = 0; k0 < KMAX; k0 += 4) {
        float4 w[4];
#pragma unroll
        for (int u = 0; u < 4; ++u)
          w[u] = k0 + u >= q.size ? make_float4(-1.f, -1.f, -1.f, -1.f) : pay[slot[k0 + u] * FTHREADS];
        piece[3 * (k0 / 4) + 0] = make_float4(w[0].y, w[0].z, w[0].w, w[1].y);
        piece[3 * (k0 / 4) + 1] = make_float4(w[1].z, w[1].w, w[2].y, w[2].z);
        piece[3 * (k0 / 4) + 2] = make_float4(w[2].w, w[3].y, w[3].z, w[3].w);
      }
      store_pair_run<3 * KMAX / 4>(reinterpret_cast<float4*>(p.bary + oa * 3), piece, odd, vA, vB);
    }
    stored = true;
   }
  }
  if (!stored && valid) {
#pragma unroll
    for (int k = 0; k < KMAX; ++k) {
      if (k < K) {
        const bool e = k >= q.size;
        const float4 w = e ? make_float4(-1.f, -1.f, -1.f, -1.f) : pay[slot[k] * FTHREADS];
        p.pix_to_face[o + k] = e ? -1ll : (long long)q.id[k];
        p.zbuf[o + k] = e ? -1.0f : q.z[k];
        p.dists[o + k] = w.x;
        p.bary[(o + k) * 3 + 0] = w.y;
        p.bary[(o + k) * 3 + 1] = w.z;
        p.bary[(o + k) * 3 + 2] = w.w;
      }
    }
  }
  if (order != ORDER_ARRIVAL || !tile_saw_tie(sh)) return;
  order = ORDER_INDEX;
  rq.reset();
  }
}

// ------------------------------------------------------------------------------------------------
// 8 < K <= 32: the same tile body with the queue keys in shared memory (SmemQueue); the winners' barycentrics
// and distances are recomputed from the face records in the epilogue (identical arithmetic, identical bits).
// Serves the reference's range of one kernel (rasterize_meshes.cu:630-736) without its 1.8 KB of thread-local
// queue per pixel.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void recompute_hit(const FineParams& p, int fi, float px, float py, Hit& h) {
  const float4* r = p.rec + (int64_t)fi * 4;
  const float4 fa = __ldg(r + 0), fb = __ldg(r + 1), fc = __ldg(r + 2);
  const Face f = {fa.x, fa.y, fc.x, fa.z, fa.w, fc.y, fb.x, fb.y, fc.z};
  eval_pixel_face<false>(px, py, f, fb.z, p.blur_radius, p.persp != 0, p.clip != 0, false, 0.0f, h);
}

template <bool NB, bool SCAN>
__global__ void __launch_bounds__(FTHREADS, 768 / FTHREADS) mesh_fine_smemq_kernel(const FineParams p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  FineStage& sh = *reinterpret_cast<FineStage*>(smem_raw);
  const int tid = threadIdx.x, lane = tid & 31;
  const TileWork t = tile_work(p);
  const int tile_x = t.tile_x, tile_y = t.tile_y, n = t.n;
  if (t.count == 0) {
    write_empty_tile<0>(p, n, tile_x, tile_y);
    return;
  }
  int xo, yo;
  fthread_pixel(tile_x, tile_y, xo, yo);
  const bool valid = xo < p.W && yo < p.H;
  const int lc = xo - tile_x * FTW, lr = yo - tile_y * FTH;
  const int K = p.K;

  SmemQueue<NB> q;
  q.init(smem_raw + sizeof(FineStage), K, tid);
  int order = first_walk_order<NB, SCAN>(t);
  for (;;) {
  fine_tile_body<SmemQueue<NB>, NB, SCAN>(p, sh, q, tile_x, tile_y, n, t.seg_begin, t.count, t.overflow, order, valid,
                                          lc, lr);
  q.sort();
  const float px = sh.col[lc], py = sh.row[lr];
  const int64_t o = (((int64_t)n * p.H + yo) * p.W + xo) * K;
  if ((K & 7) == 0) {
    // groups of 8 slots: 64 B of pix_to_face, 32 B of zbuf / dists, 96 B of barycentrics per pixel -- lanes
    // 2m / 2m+1 (adjacent pixels) write each group together, whole sectors per instruction
    const int odd = lane & 1;
    const bool vA = __shfl_sync(0xffffffffu, (int)valid, lane & ~1) != 0;
    const bool vB = __shfl_sync(0xffffffffu, (int)valid, lane | 1) != 0;
    const int64_t oa = o - (int64_t)odd * K, ob = oa + K;  // the even / odd lane's pixel
    for (int g = 0; g < K; g += 8) {
      float4 pi[4], pzv[2], pd[2], pb[6];
      float z[8], d[8], b[24];
      int id[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        Hit h = {-1.0f, -1.0f, -1.0f, -1.0f, -1.0f};
        id[u] = -1;
        if (g + u < q.size) {
          id[u] = q.qi[(g + u) * FTHREADS];
          recompute_hit(p, id[u], px, py, h);
        }
        z[u] = h.z;
        d[u] = h.dist;
        b[3 * u + 0] = h.b0;
        b[3 * u + 1] = h.b1;
        b[3 * u + 2] = h.b2;
      }
#pragma unroll
      for (int u = 0; u < 4; ++u)  // int64 = (low word, sign word)
        pi[u] = make_float4(__int_as_float(id[2 * u]), __int_as_float(id[2 * u] >> 31),
                            __int_as_float(id[2 * u + 1]), __int_as_float(id[2 * u + 1] >> 31));
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        pzv[u] = make_float4(z[4 * u], z[4 * u + 1], z[4 * u + 2], z[4 * u + 3]);
        pd[u] = make_float4(d[4 * u], d[4 * u + 1], d[4 * u + 2], d[4 * u + 3]);
      }
#pragma unroll
      for (int u = 0; u < 6; ++u) pb[u] = make_float4(b[4 * u], b[4 * u + 1], b[4 * u + 2], b[4 * u + 3]);
      store_pair_split<4>(reinterpret_cast<float4*>(p.pix_to_face + oa + g),
                          reinterpret_cast<float4*>(p.pix_to_face + ob + g), pi, odd, vA, vB);
      store_pair_split<2>(reinterpret_cast<float4*>(p.zbuf + oa + g), reinterpret_cast<float4*>(p.zbuf + ob + g), pzv,
                          odd, vA, vB);
      store_pair_split<2>(reinterpret_cast<float4*>(p.dists + oa + g), reinterpret_cast<float4*>(p.dists + ob + g),
                          pd, odd, vA, vB);
      store_pair_split<6>(reinterpret_cast<float4*>(p.bary + (oa + g) * 3),
                          reinterpret_cast<float4*>(p.bary + (ob + g) * 3), pb, odd, vA, vB);
    }
  } else if (valid) {
  for (int k = 0; k < K; ++k) {
    Hit h = {-1.0f, -1.0f, -1.0f, -1.0f, -1.0f};
    long long id = -1;
    if (k < q.size) {
      const int fi = q.qi[k * FTHREADS];
      recompute_hit(p, fi, px, py, h);
      id = fi;
    }
    p.pix_to_face[o + k] = id;
    p.zbuf[o + k] = h.z;
    p.dists[o + k] = h.dist;
    p.bary[(o + k) * 3 + 0] = h.b0;
    p.bary[(o + k) * 3 + 1] = h.b1;
    p.bary[(o + k) * 3 + 2] = h.b2;
  }
  }
  if (order != ORDER_ARRIVAL || !tile_saw_tie(sh)) return;
  order = ORDER_INDEX;
  q.reset();
  }
}

// ------------------------------------------------------------------------------------------------
// Large-K path (32 < K <= 150): the same queue in thread-local arrays holding only (z, face, dist); the
// barycentrics of the final winners are recomputed (same arithmetic, so identical values).
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(FTHREADS) mesh_fine_bigk_kernel(const FineParams p) {
  __shared__ FaceChunk s;
  const int tid = threadIdx.x, lane = tid & 31;
  const int t = blockIdx.x;
  const int n = t / (p.TY * p.TX);
  const int tile_y = (t / p.TX) % p.TY, tile_x = t % p.TX;
  int xo, yo;
  fthread_pixel(tile_x, tile_y, xo, yo);
  const bool valid = xo < p.W && yo < p.H;
  const float px = pix_to_ndc(p.W - 1 - xo, p.W, p.rx);
  const float py = pix_to_ndc(p.H - 1 - yo, p.H, p.ry);
  const float fx_lo = warp_min(valid ? px : FLT_MAX), fx_hi = warp_max(valid ? px : -FLT_MAX);
  const float fy_lo = warp_min(valid ? py : FLT_MAX), fy_hi = warp_max(valid ? py : -FLT_MAX);
  pdl_wait();
  const int seg_begin = p.tile_offset[t], seg_end = p.tile_offset[t + 1];
  const bool overflow = (int64_t)seg_end > p.capacity || seg_end == INT_MAX;
  const int64_t mesh_first = p.first[n];
  const int count = overflow ? (int)p.num[n] : seg_end - seg_begin;
  const bool persp = p.persp != 0, clip = p.clip != 0, cull = p.cull != 0;
  const int K = p.K;

  // ascending face order (see cta_sort256); the staging area doubles as the sort's scratch
  if (!overflow && count > 1)
    cta_sort_segment<FTHREADS>(p.pairs + seg_begin, count, reinterpret_cast<int*>(&s),
                               (int)(sizeof(FaceChunk) / sizeof(int)));

  float qz[B200R_MAX_K], qd[B200R_MAX_K];
  int qi[B200R_MAX_K];
  int qn = 0, q_max_idx = -1;
  float q_max_z = -1000.0f;

  for (int base = 0; base < count; base += CHUNK) {
    const int nc = min(CHUNK, count - base);
    __syncthreads();
    if (tid < nc) {
      const int f = overflow ? (int)(mesh_first + base + tid) : p.pairs[seg_begin + base + tid];
      stage_face(s, tid, p.face_verts, p.neighbor, f, p.sqrt_blur, cull);
    }
    __syncthreads();
    for (int g = 0; g < nc; g += 32) {
      bool touch = false;
      if (g + lane < nc) {
        const float4 bx = s.box[g + lane];
        touch = !(fx_lo > bx.y || fx_hi < bx.x || fy_lo > bx.w || fy_hi < bx.z);
      }
      unsigned m = __ballot_sync(0xffffffffu, touch);
      while (m) {
        const int j = g + __ffs(m) - 1;
        m &= m - 1;
        const float4 bx = s.box[j];
        if (!valid || px > bx.y || px < bx.x || py > bx.w || py < bx.z) continue;
        const float4 fa = s.a[j], fb = s.b[j], fc = s.c[j];
        const Face f = {fa.x, fa.y, fc.x, fa.z, fa.w, fc.y, fb.x, fb.y, fc.z};
        Hit h;
        const int nb = __float_as_int(fc.w);
        // (this kernel always walks sorted lists: no tie watching)
        if (!eval_pixel_face<false>(px, py, f, fb.z, p.blur_radius, persp, clip, qn >= K && nb == -1, q_max_z, h))
          continue;
        const int fi = __float_as_int(fb.w);
        int at = -1;
        if (nb != -1)
          for (int i = 0; i < qn; ++i)
            if (qi[i] == nb) {
              at = i;
              break;
            }
        if (at >= 0) {  // (:201-215)
          if (fabsf(h.dist) < fabsf(qd[at])) {
            qz[at] = h.z;
            qi[at] = fi;
            qd[at] = h.dist;
            if (h.z > q_max_z) {
              q_max_z = h.z;
              q_max_idx = at;
            }
          }
        } else if (qn < K) {  // (:218-225)
          qz[qn] = h.z;
          qi[qn] = fi;
          qd[qn] = h.dist;
          if (h.z > q_max_z) {
            q_max_z = h.z;
            q_max_idx = qn;
          }
          ++qn;
        } else if (h.z < q_max_z) {  // (:226-236)
          qz[q_max_idx] = h.z;
          qi[q_max_idx] = fi;
          qd[q_max_idx] = h.dist;
          q_max_z = h.z;
          for (int i = 0; i < K; ++i)
            if (qz[i] > q_max_z) {
              q_max_z = qz[i];
              q_max_idx = i;
            }
        }
      }
    }
  }
  if (!valid) return;
  // sort by (z, face): insertion sort, keys unique
  for (int i = 1; i < qn; ++i) {
    const float tz = qz[i];
    const int ti = qi[i];
    int j = i - 1;
    while (j >= 0 && key_less(tz, ti, qz[j], qi[j])) {
      qz[j + 1] = qz[j];
      qi[j + 1] = qi[j];
      --j;
    }
    qz[j + 1] = tz;
    qi[j + 1] = ti;
  }
  const int64_t o = (((int64_t)n * p.H + yo) * p.W + xo) * K;
  for (int k = 0; k < K; ++k) {
    Hit h = {-1.0f, -1.0f, -1.0f, -1.0f, -1.0f};
    long long id = -1;
    if (k < qn) {
      const float* v = p.face_verts + (int64_t)qi[k] * 9;
      const Face f = {__ldg(v + 0), __ldg(v + 1), __ldg(v + 2), __ldg(v + 3), __ldg(v + 4),
                      __ldg(v + 5), __ldg(v + 6), __ldg(v + 7), __ldg(v + 8)};
      eval_pixel_face<false>(px, py, f, bary_denominator(f), p.blur_radius, persp, clip, false, 0.0f, h);
      id = qi[k];
    }
    p.pix_to_face[o + k] = id;
    p.zbuf[o + k] = h.z;
    p.dists[o + k] = h.dist;
    p.bary[(o + k) * 3 + 0] = h.b0;
    p.bary[(o + k) * 3 + 1] = h.b1;
    p.bary[(o + k) * 3 + 2] = h.b2;
  }
}

// ------------------------------------------------------------------------------------------------
// Backward: one thread per pixel (same 16x16 tiles / 8x4 warp footprints as the forward pass, so the
// faces a warp scatters into are spatially coherent), chain rule of rasterize_meshes.cu:466-561 with
// BarycentricClipBackward fed the perspective-corrected barycentrics like the forward pass and the
// CPU implementation (rasterize_meshes_cpu.cpp:498-500).
// ------------------------------------------------------------------------------------------------
struct BackwardParams {
  const float* face_verts;
  const int64_t* pix_to_face;
  const float* grad_zbuf;
  const float* grad_bary;
  const float* grad_dists;
  int N, H, W, K, TY, TX;
  int n0;  // first image of this launch
  int g_vec;   // the gradient output is 8-byte aligned: 8-byte vector reductions
  int64_t F;
  float rx, ry;
  int persp, clip;
  float* grad_face_verts;
  // fused entry point: the per-face gradient goes straight into the vertices (grad_verts[faces[f][j]]) -- what the
  // backward of `verts_packed[faces_packed]` does -- instead of into grad_face_verts followed by a scatter pass
  const int64_t* faces;  // nullptr: plain (F,3,3) output
  float* grad_verts;
  int64_t V;
};

__device__ __forceinline__ void edge_bwd(float px, float py, float ax, float ay, float bx, float by, float g,
                                         float2& dp, float2& da, float2& db) {
  dp = make_float2(g * (by - ay), g * (ax - bx));
  da = make_float2(g * (py - by), g * (bx - px));
  db = make_float2(g * (ay - py), g * (px - ax));
}

__device__ __forceinline__ void point_line_bwd(float px, float py, float ax, float ay, float bx, float by, float g,
                                               float2& ga, float2& gb) {
  const float bax = bx - ax, bay = by - ay;
  const float t = __saturatef((bax * (px - ax) + bay * (py - ay)) / (bax * bax + bay * bay));
  const float qx = (1.0f - t) * ax + t * bx, qy = (1.0f - t) * ay + t * by;
  const float cx = 2.0f * (qx - px), cy = 2.0f * (qy - py);
  ga = make_float2(g * (1.0f - t) * cx, g * (1.0f - t) * cy);
  gb = make_float2(g * t * cx, g * t * cy);
}

// Gradient of one (pixel, face) hit with respect to the face's 9 coordinates (out[0..8]).
__device__ __forceinline__ void backward_one(const BackwardParams& p, float px, float py, int64_t fi, float gz,
                                             float gd, float gb0, float gb1, float gb2, bool persp, bool clip,
                                             float (&out)[9]) {
  const float* v = p.face_verts + fi * 9;
  // (the face's 36 bytes as the three 16-byte pieces that contain them, shifted into place with selects -- 3 load
  // instructions instead of 9 -- was measured and is no gain: north-star batch 94.2 vs 94.2 us, with blur 222 vs 215 us)
  const Face f = {__ldg(v + 0), __ldg(v + 1), __ldg(v + 2), __ldg(v + 3), __ldg(v + 4),
                  __ldg(v + 5), __ldg(v + 6), __ldg(v + 7), __ldg(v + 8)};
  const float den = bary_denominator(f);
  float w0, w1, w2;
  bary_coords(px, py, f, den, w0, w1, w2);
  float c0 = w0, c1 = w1, c2 = w2;  // (perspective-corrected) barycentrics
  if (persp) bary_persp(c0, c1, c2, f.z0, f.z1, f.z2);
  float k0 = c0, k1 = c1, k2 = c2;  // clipped
  if (clip) bary_clip(k0, k1, k2);
  const bool inside = c0 > 0.0f && c1 > 0.0f && c2 > 0.0f;
  const float sgd = inside ? -gd : gd;

  // d dist / d verts: gradient flows to the closest edge only (geometry_utils.cuh:421-462)
  float2 dv0 = make_float2(0.f, 0.f), dv1 = dv0, dv2 = dv0;
  {
    const float e01 = point_line_dist(px, py, f.x0, f.y0, f.x1, f.y1);
    const float e02 = point_line_dist(px, py, f.x0, f.y0, f.x2, f.y2);
    const float e12 = point_line_dist(px, py, f.x1, f.y1, f.x2, f.y2);
    if (e01 <= e02 && e01 <= e12)
      point_line_bwd(px, py, f.x0, f.y0, f.x1, f.y1, sgd, dv0, dv1);
    else if (e02 <= e01 && e02 <= e12)
      point_line_bwd(px, py, f.x0, f.y0, f.x2, f.y2, sgd, dv0, dv2);
    else if (e12 <= e01 && e12 <= e02)
      point_line_bwd(px, py, f.x1, f.y1, f.x2, f.y2, sgd, dv1, dv2);
  }

  // upstream gradient on the (clipped) barycentrics, including zbuf = sum_i bary_i * z_i
  float g0 = gb0 + gz * f.z0, g1 = gb1 + gz * f.z1, g2 = gb2 + gz * f.z2;
  if (clip) {  // BarycentricClipBackward (geometry_utils.cuh:273-329) on the corrected barycentrics
    const float m0 = fmaxf(c0, 0.0f), m1 = fmaxf(c1, 0.0f), m2 = fmaxf(c2, 0.0f);
    float sum = m0 + m1 + m2, gsc = 1.0f;
    if (sum < 1e-5f) {
      gsc = 0.0f;
      sum = 1e-5f;
    }
    const float inv = __frcp_rn(sum), inv2 = gsc * inv * inv;
    const float s0 = -m0 * inv2, s1 = -m1 * inv2, s2 = -m2 * inv2;
    const float cross = g0 * s0 + g1 * s1 + g2 * s2;
    const float n0 = c0 < 0.0f ? 0.0f : g0 * inv + cross;
    const float n1 = c1 < 0.0f ? 0.0f : g1 * inv + cross;
    const float n2 = c2 < 0.0f ? 0.0f : g2 * inv + cross;
    g0 = n0;
    g1 = n1;
    g2 = n2;
  }
  float dz0 = 0.0f, dz1 = 0.0f, dz2 = 0.0f;
  if (persp) {  // BarycentricPerspectiveCorrectionBackward (geometry_utils.cuh:200-228)
    const float t0 = w0 * f.z1 * f.z2, t1 = f.z0 * w1 * f.z2, t2 = f.z0 * f.z1 * w2;
    const float dn = fmaxf(t0 + t1 + t2, 1e-8f);
    const float rdn = __frcp_rn(dn);
    const float gdn = (-t0 * g0 - t1 * g1 - t2 * g2) * rdn * rdn;
    const float h0 = gdn + g0 * rdn, h1 = gdn + g1 * rdn, h2 = gdn + g2 * rdn;
    g0 = h0 * f.z1 * f.z2;
    g1 = h1 * f.z0 * f.z2;
    g2 = h2 * f.z0 * f.z1;
    dz0 = h1 * w1 * f.z2 + h2 * w2 * f.z1;
    dz1 = h0 * w0 * f.z2 + h2 * w2 * f.z0;
    dz2 = h0 * w0 * f.z1 + h1 * w1 * f.z0;
  }
  // BarycentricCoordsBackward (geometry_utils.cuh:101-161)
  float2 bv0 = make_float2(0.f, 0.f), bv1 = bv0, bv2 = bv0;
  {
    const float rden = __frcp_rn(den);
    const float e0 = edge_fn(px, py, f.x1, f.y1, f.x2, f.y2);
    const float e1 = edge_fn(px, py, f.x2, f.y2, f.x0, f.y0);
    const float e2 = edge_fn(px, py, f.x0, f.y0, f.x1, f.y1);
    float2 dp, da, db, ap, aa, ab;
    // every w_i = e_i / area also depends on area = E(v2; v0, v1)
    const float garea = -(g0 * e0 + g1 * e1 + g2 * e2) * rden * rden;
    edge_bwd(f.x2, f.y2, f.x0, f.y0, f.x1, f.y1, garea, ap, aa, ab);  // (p=v2, a=v0, b=v1)
    bv2.x += ap.x; bv2.y += ap.y;
    bv0.x += aa.x; bv0.y += aa.y;
    bv1.x += ab.x; bv1.y += ab.y;
    edge_bwd(px, py, f.x1, f.y1, f.x2, f.y2, g0 * rden, dp, da, db);  // w0: (p, v1, v2)
    bv1.x += da.x; bv1.y += da.y;
    bv2.x += db.x; bv2.y += db.y;
    edge_bwd(px, py, f.x2, f.y2, f.x0, f.y0, g1 * rden, dp, da, db);  // w1: (p, v2, v0)
    bv2.x += da.x; bv2.y += da.y;
    bv0.x += db.x; bv0.y += db.y;
    edge_bwd(px, py, f.x0, f.y0, f.x1, f.y1, g2 * rden, dp, da, db);  // w2: (p, v0, v1)
    bv0.x += da.x; bv0.y += da.y;
    bv1.x += db.x; bv1.y += db.y;
  }
  out[0] = bv0.x + dv0.x;
  out[1] = bv0.y + dv0.y;
  out[2] = gz * k0 + dz0;
  out[3] = bv1.x + dv1.x;
  out[4] = bv1.y + dv1.y;
  out[5] = gz * k1 + dz1;
  out[6] = bv2.x + dv2.x;
  out[7] = bv2.y + dv2.y;
  out[8] = gz * k2 + dz2;
}

// Scatter one warp's contributions.  Neighbouring pixels usually hit the same face, so before touching memory
// the warp merges ALL lanes that carry the same face: one set of 9 atomics per distinct face of the warp
// instead of per pixel (the kernel is sensitive to the number of atomics: merging only within pixel rows costs
// +10 us on the north-star batch).
__device__ __forceinline__ void red_add_v2(float* addr, float a, float b) {  // sm_90+ vector reduction, 8-byte aligned
  asm volatile("red.global.add.v2.f32 [%0], {%1, %2};" ::"l"(addr), "f"(a), "f"(b) : "memory");
}
__device__ __forceinline__ void warp_scatter(const BackwardParams& p, int face, float (&g)[9], int lane) {
  // All lanes that hit the same face are found with one MATCH; each lane then adds up its successors in the
  // group by pointer jumping (after round r a lane holds the sum of 2^r consecutive group members), so the
  // group's lowest lane ends up with the whole sum after ceil(log2(group size)) rounds -- typically one or
  // two, faces being a few pixels large -- and is the only one to issue atomics.
  const unsigned grp = __match_any_sync(0xffffffffu, face);
  const unsigned above = lane == 31 ? 0u : grp & (0xffffffffu << (lane + 1));
  int next = (face >= 0 && above != 0u) ? __ffs((int)above) - 1 : -1;
  while (__any_sync(0xffffffffu, next >= 0)) {
    const int src = next >= 0 ? next : lane;
#pragma unroll
    for (int i = 0; i < 9; ++i) {
      const float v = __shfl_sync(0xffffffffu, g[i], src);
      if (next >= 0) g[i] += v;
    }
    const int nn = __shfl_sync(0xffffffffu, next, src);
    next = next >= 0 ? nn : -1;
  }
  // (runs of consecutive lanes with the same face -- a shuffle and a vote instead of MATCH, with a segmented shuffle-down
  // reduction -- were measured against this: 96.3 vs 94.2 us, with blur 249 vs 215 us: faces span pixel rows)
  if (face >= 0 && lane == __ffs((int)grp) - 1) {
    // (the kernel is sensitive to the number of reduction instructions -- with a blur band, where most slots are hits, they
    // bound it: north-star batch with blur 1e-4 280 -> 222 us, config 5 447 -> 344 us with 8-byte vector reductions where
    // the target is 8-byte aligned: a face's 36 bytes / a vertex's 12 bytes start at a multiple of 4 whose parity is that
    // of the index; 5 instead of 9 / 6 instead of 9 instructions, the same words and sums)
    if (p.faces != nullptr) {
      const int64_t* fc = p.faces + (int64_t)face * 3;
#pragma unroll
      for (int j = 0; j < 3; ++j) {
        const int64_t vi = __ldg(fc + j);
        if (vi < 0 || vi >= p.V) continue;  // (out-of-range indices: an error in the reference; ignored like the gather)
        float* o = p.grad_verts + vi * 3;
        if (p.g_vec) {
          const bool odd = (vi & 1) != 0;
          const float s1 = odd ? g[3 * j] : g[3 * j + 2];
          const float a = odd ? g[3 * j + 1] : g[3 * j], b = odd ? g[3 * j + 2] : g[3 * j + 1];
          if (s1 != 0.0f) atomicAdd(o + (odd ? 0 : 2), s1);
          if (a != 0.0f || b != 0.0f) red_add_v2(o + (odd ? 1 : 0), a, b);
          continue;
        }
#pragma unroll
        for (int c = 0; c < 3; ++c)
          if (g[3 * j + c] != 0.0f) atomicAdd(o + c, g[3 * j + c]);
      }
    } else {
      float* o = p.grad_face_verts + (int64_t)face * 9;
      // (16-byte reductions on the aligned groups inside the 36 bytes -- a four-way switch on face & 3, 3 or 4 reductions per
      // face -- were measured against this: north-star batch with blur 225 vs 215 us, config 5 364 vs 354 us: the divergent
      // switch costs more than the shorter sequences save)
      if (p.g_vec) {
        const int odd = face & 1;
        atomicAdd(o + (odd ? 0 : 8), odd ? g[0] : g[8]);
#pragma unroll
        for (int j = 0; j < 4; ++j)
          red_add_v2(o + 2 * j + odd, odd ? g[2 * j + 1] : g[2 * j], odd ? g[2 * j + 2] : g[2 * j + 1]);
        return;
      }
#pragma unroll
      for (int i = 0; i < 9; ++i) atomicAdd(o + i, g[i]);
    }
  }
}

// GV > 0: K is a multiple of GV (8 or 4) and a pixel's face indices are fetched GV at a time with 16-byte loads
// (a group without faces costs nothing else); GV == 0: any K, scalar loads.
// Resident CTAs per SM the register budget is set for.  (Measured on the north-star batch: 4 CTAs, 64 registers: 96.3 us;
// 5 CTAs, 48 registers, 84 bytes of spills: 135.2 us; 6 CTAs, 40 registers: 163.9 us -- the kernel is bound by load/store
// instructions through the L1 pipeline, not by the warps in flight: every spill is one more of them.  For the same reason
// pulling the next wave's indices into L2 with prefetch instructions -- `prefetch.global.L2` of the tile one wave of CTAs
// ahead -- costs 96.3 -> 100.4 us, and an L1 prefetch of the next slot's face 96.3 -> 100.4 us.  Fetching the upstream
// gradients of a pixel's first four slots with five 16-byte loads as soon as the indices are known -- one DRAM round trip
// instead of one per slot -- needs 80 registers, three CTAs: 96 -> 113 us.)
constexpr int BWD_CTAS = 4;
template <int GV>
__global__ void __launch_bounds__(TILE_THREADS, BWD_CTAS) mesh_backward_kernel(const BackwardParams p) {
  const int lane = threadIdx.x & 31;
  const int tile_x = blockIdx.x, tile_y = blockIdx.y, n = p.n0 + blockIdx.z;  // grid = (TX, TY, images)
  int xo, yo;
  thread_pixel(tile_x, tile_y, xo, yo);
  const bool in_image = xo < p.W && yo < p.H;
  const float px = pix_to_ndc(p.W - 1 - xo, p.W, p.rx);
  const float py = pix_to_ndc(p.H - 1 - yo, p.H, p.ry);
  const int K = p.K;
  const int64_t o = in_image ? (((int64_t)n * p.H + yo) * p.W + xo) * K : 0;
  const bool persp = p.persp != 0, clip = p.clip != 0;
  constexpr int G = GV > 0 ? GV : 1;

  for (int k0 = 0; k0 < K; k0 += G) {
    int fk[G];
    if (GV > 0) {
#pragma unroll
      for (int k = 0; k < G; k += 2) {
        longlong2 v = make_longlong2(-1, -1);
        if (in_image) v = __ldg(reinterpret_cast<const longlong2*>(p.pix_to_face + o + k0 + k));
        fk[k] = (int)v.x;  // the reference reads the int64 index into an int as well (:471)
        fk[k + 1] = (int)v.y;
      }
    } else {
      fk[0] = in_image ? (int)p.pix_to_face[o + k0] : -1;
    }
#pragma unroll 1
    for (int j = 0; j < G; ++j) {
      const int face = fk[0];
#pragma unroll
      for (int u = 0; u + 1 < G; ++u) fk[u] = fk[u + 1];  // rotate: one copy of the gradient code
      if (!__any_sync(0xffffffffu, face >= 0)) continue;  // padded slots (:472-474)
      float g[9] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
      if (face >= 0) {
        const int64_t i = o + k0 + j;
        const float gz = __ldg(p.grad_zbuf + i);
        const float gd = __ldg(p.grad_dists + i);
        // (8 + 4 byte loads of the three barycentric gradients instead of three scalar ones: 94.2 -> 98.4 us, more spills)
        const float gb0 = __ldg(p.grad_bary + i * 3);
        const float gb1 = __ldg(p.grad_bary + i * 3 + 1);
        const float gb2 = __ldg(p.grad_bary + i * 3 + 2);
        backward_one(p, px, py, face, gz, gd, gb0, gb1, gb2, persp, clip, g);
      }
      warp_scatter(p, face, g, lane);
    }
  }
}

}  // namespace b200r

// The face gather alone (only used when there is no image to rasterize): what `verts_packed[faces_packed]` does
// (rasterize_meshes.py:144-148); its backward -- the scatter-add into the vertices -- is part of the backward kernel.
__global__ void __launch_bounds__(256) mesh_gather_kernel(const float* __restrict__ verts, int64_t V,
                                                          const int64_t* __restrict__ faces, int64_t F,
                                                          float* __restrict__ face_verts_out) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;  // (face, corner)
  if (e >= F * 3) return;
  const int64_t vi = __ldg(faces + e);
  const bool ok = vi >= 0 && vi < V;
#pragma unroll
  for (int c = 0; c < 3; ++c) face_verts_out[e * 3 + c] = ok ? __ldg(verts + vi * 3 + c) : __int_as_float(0x7fc00000);
}

// ================================================================================================
// C ABI
// ================================================================================================
using namespace b200r;

extern "C" size_t b200r_rasterize_meshes_workspace_bytes(int64_t F, int32_t N, int32_t H, int32_t W,
                                                         int64_t pair_capacity) {
  if (F < 0 || N < 0 || H < 0 || W < 0) return 0;
  return carve_workspace(nullptr, F, N, H, W, pair_capacity, FTH, FTW).bytes +
         FACE_RECORD_BYTES * (size_t)(F > 0 ? F : 1);
}

static int forward_impl(const float* face_verts, const float* verts, int64_t V, const int64_t* faces,
                        float* face_verts_out, int64_t F, const int64_t* first, const int64_t* num,
                        const int64_t* neighbor, int32_t N, int32_t H, int32_t W, float blur_radius, int32_t K,
                        int32_t perspective_correct, int32_t clip_barycentric_coords, int32_t cull_backfaces,
                        int64_t* pix_to_face, float* zbuf, float* bary, float* dists, void* workspace,
                        size_t workspace_bytes, int64_t pair_capacity, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  if (K > B200R_MAX_K) return fail(B200R_ERR_INVALID_ARGUMENT, "Must have points_per_pixel <= 150");
  if (F < 0 || N < 0 || H < 0 || W < 0 || K < 0) return fail(B200R_ERR_INVALID_ARGUMENT, "negative size");
  if (F > INT_MAX) return fail(B200R_ERR_INVALID_ARGUMENT, "more than 2^31-1 packed faces are not supported");
  if ((int64_t)N * H * W * K == 0) return B200R_OK;  // empty outputs (rasterize_meshes.cu:793-796)
  const int TY = div_up(H, FTH), TX = div_up(W, FTW);
  if (TY > 0xFFFE || TX > 0xFFFE) return fail(B200R_ERR_INVALID_ARGUMENT, "image too large");
  const int64_t ntiles = (int64_t)N * TY * TX;
  if (ntiles > INT_MAX) return fail(B200R_ERR_INVALID_ARGUMENT, "too many tiles");
  BinWorkspace ws = carve_workspace(workspace, F, N, H, W, pair_capacity, FTH, FTW);
  const size_t nrec = (size_t)(F > 0 ? F : 1);
  if (workspace == nullptr || workspace_bytes < ws.bytes + FACE_RECORD_BYTES * nrec)
    return fail(B200R_ERR_WORKSPACE, "workspace too small for rasterize_meshes_forward");
  float4* rec = reinterpret_cast<float4*>(static_cast<char*>(workspace) + ws.bytes);  // (ws.bytes % 16 == 0)

  const float rx = ndc_range(W, H), ry = ndc_range(H, W);
  const float sqrt_blur = sqrtf(blur_radius);  // IEEE sqrt, like the device sqrt.rn of the reference

  const bool prof = profiling_enabled();
  if (prof) phase_timer().record(0, stream);
  zero_ints_kernel<<<(unsigned)((ntiles + 1023) / 1024), 256, 0, stream>>>(ws.tile_count, ntiles);
  B200R_LAUNCHED("zero_ints_kernel");
  if (F > 0) {
    const dim3 sgrid((unsigned)((F + SETUP_FACES - 1) / SETUP_FACES));
    if (faces != nullptr) {
      B200R_CUDA_OK(launch_chained(mesh_setup_count_kernel<true>, sgrid, dim3(SETUP_FACES), 0, stream,
                                   (const float*)nullptr, verts, V, faces, face_verts_out, neighbor, F, first, num, N, H,
                                   W, TY, TX, rx, ry, sqrt_blur, cull_backfaces, ws.rect, ws.tile_count, rec));
      face_verts = face_verts_out;
    } else {
      B200R_CUDA_OK(launch_chained(mesh_setup_count_kernel<false>, sgrid, dim3(SETUP_FACES), 0, stream, face_verts,
                                   (const float*)nullptr, (int64_t)0, (const int64_t*)nullptr, (float*)nullptr,
                                   neighbor, F, first, num, N, H, W, TY, TX, rx, ry, sqrt_blur, cull_backfaces, ws.rect,
                                   ws.tile_count, rec));
    }
    B200R_LAUNCHED("mesh_setup_count_kernel");
  }
  // Schedule of the fine pass (see tile_scan_kernel): worth the extra pass of the scan kernel and one more dependent load
  // per CTA where tiles run long -- with a blur band (north-star batch + blur 1e-4: fine 918 -> 749 us, config 2: 137 ->
  // 109 us); without one the north-star batch loses 6 us.  The packed class counters hold 2^21 tiles.
  int* const tile_order = (blur_radius > 0.0f && ntiles < (1ll << ORDER_BITS)) ? ws.tile_order : nullptr;
  B200R_CUDA_OK(launch_chained(tile_scan_kernel, dim3(1), dim3(1024), 0, stream, ws.tile_count, ws.tile_offset,
                               (int)ntiles, tile_order));
  B200R_LAUNCHED("tile_scan_kernel");
  if (F > 0) {
    B200R_CUDA_OK(launch_chained(tile_fill_kernel<true>, dim3((unsigned)((F + 255) / 256)), dim3(256), 0, stream,
                                 ws.rect, F, TY, TX, ws.tile_count, ws.pairs, ws.capacity));
    B200R_LAUNCHED("tile_fill_kernel");
  }
  // (no sort launch: every fine CTA puts its own tile list in ascending face order, see cta_sort256)
  if (prof) phase_timer().record(1, stream);
  FineParams p;
  p.face_verts = face_verts;
  p.neighbor = neighbor;
  p.rec = rec;
  p.n0 = 0;
  p.first = first;
  p.num = num;
  p.tile_offset = ws.tile_offset;
  p.tile_order = tile_order;
  p.pairs = ws.pairs;
  p.capacity = ws.capacity;
  p.N = N; p.H = H; p.W = W; p.K = K; p.TY = TY; p.TX = TX;
  p.rx = rx; p.ry = ry; p.blur_radius = blur_radius; p.sqrt_blur = sqrt_blur;
  p.persp = perspective_correct; p.clip = clip_barycentric_coords; p.cull = cull_backfaces;
  p.smem_ints = 0;
  p.pix_to_face = pix_to_face; p.zbuf = zbuf; p.bary = bary; p.dists = dists;
  const unsigned grid = (unsigned)ntiles;
  const bool no_blur = !(blur_radius > 0.0f);
  int dev_ = 0;
  B200R_CUDA_OK(cudaGetDevice(&dev_));
  // > 48 KB of dynamic shared memory: opt-in once per kernel and device
#define B200R_FINE_LAUNCH(KERNEL, SMEM_MAX, SMEM)                                                         \
  do {                                                                                                   \
    static bool configured[64] = {};                                                                     \
    if (dev_ < 0 || dev_ >= 64 || !configured[dev_]) {                                                   \
      B200R_CUDA_OK(cudaFuncSetAttribute(KERNEL, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(SMEM_MAX))); \
      if (dev_ >= 0 && dev_ < 64) configured[dev_] = true;                                               \
    }                                                                                                    \
    p.smem_ints = (int)((SMEM) / sizeof(int));                                                           \
    for (p.n0 = 0; p.n0 < N; p.n0 += 65535) {                                                            \
      const dim3 grid3((unsigned)TX, (unsigned)TY, (unsigned)min(N - p.n0, 65535));                      \
      B200R_CUDA_OK(launch_chained(KERNEL, grid3, dim3(FTHREADS), (SMEM), stream, p));                   \
    }                                                                                                    \
  } while (0)
#define B200R_FINE(KM)                                                                                    \
  do {                                                                                                   \
    constexpr size_t smem_ = sizeof(FineStage) + sizeof(float4) * KM * FTHREADS;                         \
    if (neighbor && no_blur)                                                                             \
      B200R_FINE_LAUNCH((mesh_fine_kernel<KM, true, true>), smem_, smem_);                               \
    else if (neighbor)                                                                                   \
      B200R_FINE_LAUNCH((mesh_fine_kernel<KM, true, false>), smem_, smem_);                              \
    else if (no_blur)                                                                                    \
      B200R_FINE_LAUNCH((mesh_fine_kernel<KM, false, true>), smem_, smem_);                              \
    else                                                                                                 \
      B200R_FINE_LAUNCH((mesh_fine_kernel<KM, false, false>), smem_, smem_);                             \
  } while (0)
  if (K <= 1)
    B200R_FINE(1);
  else if (K <= 2)
    B200R_FINE(2);
  else if (K <= 4)
    B200R_FINE(4);
  else if (K <= 8)
    B200R_FINE(8);
  else if (K <= SMEMQ_MAX_K) {
    // queue keys in shared memory: (z, face) per slot, plus the signed distance for the neighbour rule
    const size_t smem_max_nb = sizeof(FineStage) + (size_t)SMEMQ_MAX_K * FTHREADS * 12;
    const size_t smem_max = sizeof(FineStage) + (size_t)SMEMQ_MAX_K * FTHREADS * 8;
    const size_t smem_nb = sizeof(FineStage) + (size_t)K * FTHREADS * 12;
    const size_t smem = sizeof(FineStage) + (size_t)K * FTHREADS * 8;
    if (neighbor && no_blur)
      B200R_FINE_LAUNCH((mesh_fine_smemq_kernel<true, true>), smem_max_nb, smem_nb);
    else if (neighbor)
      B200R_FINE_LAUNCH((mesh_fine_smemq_kernel<true, false>), smem_max_nb, smem_nb);
    else if (no_blur)
      B200R_FINE_LAUNCH((mesh_fine_smemq_kernel<false, true>), smem_max, smem);
    else
      B200R_FINE_LAUNCH((mesh_fine_smemq_kernel<false, false>), smem_max, smem);
  } else
    B200R_CUDA_OK(launch_chained(mesh_fine_bigk_kernel, dim3(grid), dim3(FTHREADS), 0, stream, p));
#undef B200R_FINE
#undef B200R_FINE_LAUNCH
  B200R_LAUNCHED("mesh_fine_kernel");
  if (prof) {
    phase_timer().record(2, stream);
    phase_timer().have_fwd = true;
  }
  return B200R_OK;
}

extern "C" int b200r_rasterize_meshes_forward(const float* face_verts, int64_t F, const int64_t* first,
                                              const int64_t* num, const int64_t* neighbor, int32_t N, int32_t H,
                                              int32_t W, float blur_radius, int32_t K, int32_t bin_size,
                                              int32_t max_faces_per_bin, int32_t perspective_correct,
                                              int32_t clip_barycentric_coords, int32_t cull_backfaces,
                                              int64_t* pix_to_face, float* zbuf, float* bary, float* dists,
                                              void* workspace, size_t workspace_bytes, int64_t pair_capacity,
                                              void* stream_) {
  (void)bin_size;
  (void)max_faces_per_bin;
  return forward_impl(face_verts, nullptr, 0, nullptr, nullptr, F, first, num, neighbor, N, H, W, blur_radius, K,
                      perspective_correct, clip_barycentric_coords, cull_backfaces, pix_to_face, zbuf, bary, dists,
                      workspace, workspace_bytes, pair_capacity, stream_);
}

extern "C" int b200r_rasterize_meshes_forward_indexed(const float* verts, int64_t V, const int64_t* faces, int64_t F,
                                                      const int64_t* first, const int64_t* num,
                                                      const int64_t* neighbor, int32_t N, int32_t H, int32_t W,
                                                      float blur_radius, int32_t K, int32_t perspective_correct,
                                                      int32_t clip_barycentric_coords, int32_t cull_backfaces,
                                                      int64_t* pix_to_face, float* zbuf, float* bary, float* dists,
                                                      float* face_verts_out, void* workspace,
                                                      size_t workspace_bytes, int64_t pair_capacity,
                                                      void* stream_) {
  if (V < 0) return fail(B200R_ERR_INVALID_ARGUMENT, "negative size");
  if (F > 0 && (faces == nullptr || face_verts_out == nullptr || (V > 0 && verts == nullptr)))
    return fail(B200R_ERR_INVALID_ARGUMENT, "verts, faces and face_verts_out must not be null");
  if ((int64_t)N * H * W * K == 0 && F > 0) {
    // no image to produce, but the gathered faces are still an output
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    mesh_gather_kernel<<<(unsigned)((F * 3 + 255) / 256), 256, 0, stream>>>(verts, V, faces, F, face_verts_out);
    B200R_LAUNCHED("mesh_gather_kernel");
    return B200R_OK;
  }
  return forward_impl(nullptr, verts, V, F > 0 ? faces : nullptr, face_verts_out, F, first, num, neighbor, N, H, W,
                      blur_radius, K, perspective_correct, clip_barycentric_coords, cull_backfaces, pix_to_face,
                      zbuf, bary, dists, workspace, workspace_bytes, pair_capacity, stream_);
}

static int backward_impl(const float* face_verts, int64_t F, const int64_t* pix_to_face, const float* grad_zbuf,
                         const float* grad_bary, const float* grad_dists, int32_t N, int32_t H, int32_t W, int32_t K,
                         int32_t perspective_correct, int32_t clip_barycentric_coords, float* grad_face_verts,
                         const int64_t* faces, float* grad_verts, int64_t V, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  if (F < 0 || N < 0 || H < 0 || W < 0 || K < 0) return fail(B200R_ERR_INVALID_ARGUMENT, "negative size");
  if (F == 0) return B200R_OK;
  if (faces == nullptr) B200R_CUDA_OK(cudaMemsetAsync(grad_face_verts, 0, sizeof(float) * 9 * (size_t)F, stream));
  if ((int64_t)N * H * W * K == 0) return B200R_OK;
  const int TY = div_up(H, TILE), TX = div_up(W, TILE);
  BackwardParams p;
  p.face_verts = face_verts; p.pix_to_face = pix_to_face;
  p.grad_zbuf = grad_zbuf; p.grad_bary = grad_bary; p.grad_dists = grad_dists;
  p.N = N; p.H = H; p.W = W; p.K = K; p.TY = TY; p.TX = TX;
  p.F = F;
  p.g_vec = (reinterpret_cast<uintptr_t>(faces != nullptr ? grad_verts : grad_face_verts) & 7u) == 0 ? 1 : 0;
  p.rx = ndc_range(W, H); p.ry = ndc_range(H, W);
  p.persp = perspective_correct; p.clip = clip_barycentric_coords;
  p.grad_face_verts = grad_face_verts;
  p.faces = faces;
  p.grad_verts = grad_verts;
  p.V = V;
  const bool prof = profiling_enabled();
  if (prof) phase_timer().record(3, stream);
  for (p.n0 = 0; p.n0 < N; p.n0 += 65535) {  // grid.z is limited to 65535 images per launch
    const dim3 bgrid((unsigned)TX, (unsigned)TY, (unsigned)min(N - p.n0, 65535));
    if ((K & 7) == 0)
      mesh_backward_kernel<8><<<bgrid, TILE_THREADS, 0, stream>>>(p);
    else if ((K & 3) == 0)
      mesh_backward_kernel<4><<<bgrid, TILE_THREADS, 0, stream>>>(p);
    else
      mesh_backward_kernel<0><<<bgrid, TILE_THREADS, 0, stream>>>(p);
  }
  B200R_LAUNCHED("mesh_backward_kernel");
  if (prof) {
    phase_timer().record(4, stream);
    phase_timer().have_bwd = true;
  }
  return B200R_OK;
}

extern "C" int b200r_rasterize_meshes_backward(const float* face_verts, int64_t F, const int64_t* pix_to_face,
                                               const float* grad_zbuf, const float* grad_bary,
                                               const float* grad_dists, int32_t N, int32_t H, int32_t W, int32_t K,
                                               int32_t perspective_correct, int32_t clip_barycentric_coords,
                                               float* grad_face_verts, void* stream_) {
  return backward_impl(face_verts, F, pix_to_face, grad_zbuf, grad_bary, grad_dists, N, H, W, K, perspective_correct,
                       clip_barycentric_coords, grad_face_verts, nullptr, nullptr, 0, stream_);
}

extern "C" int b200r_rasterize_meshes_backward_indexed(const float* face_verts, const int64_t* faces, int64_t F,
                                                       int64_t V, const int64_t* pix_to_face,
                                                       const float* grad_zbuf, const float* grad_bary,
                                                       const float* grad_dists, int32_t N, int32_t H, int32_t W,
                                                       int32_t K, int32_t perspective_correct,
                                                       int32_t clip_barycentric_coords, float* grad_verts,
                                                       float* grad_face_verts_scratch, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  if (F < 0 || V < 0) return fail(B200R_ERR_INVALID_ARGUMENT, "negative size");
  if (V > 0) B200R_CUDA_OK(cudaMemsetAsync(grad_verts, 0, sizeof(float) * 3 * (size_t)V, stream));
  if (F == 0 || V == 0) return B200R_OK;
  // (the kernel adds every group's gradient straight to the three vertices of its face: no (F,3,3) intermediate and
  // no scatter pass -- 20 MB written and read again and one launch less per step at the north-star size;
  // `grad_face_verts_scratch` is no longer touched)
  (void)grad_face_verts_scratch;
  return backward_impl(face_verts, F, pix_to_face, grad_zbuf, grad_bary, grad_dists, N, H, W, K, perspective_correct,
                       clip_barycentric_coords, nullptr, faces, grad_verts, V, stream_);
}
