// bvh_device.cu -- the bvh.js tree (bvh_builder.cpp's output, bit for bit) built on the GPU: fspt_bvh_build_device.
//
// Every split decision of bvh.js is exact binary64 arithmetic (bvh_sah.h, shared with the host builder) and node boxes are
// unions under a total order, so any grouping of the same unions gives the same doubles.  The build is top-down and
// level-synchronous:
//   1. per-triangle boxes (stale `tb` for presorts and sweeps, current `nb` for node boxes) and centroid sort keys;
//   2. three stable presorts: LSD radix sort of 64-bit order-preserving keys (-0.0 mapped to +0.0 first, because the host's
//      `cc[p] < cc[q]` treats the two as equal) with the triangle index as payload;
//   3. one level at a time, every segment [lo, hi) of more than kSmall triangles is cut into chunks of kChunk positions:
//      chunk unions -> per-segment prefix / suffix over the chunks -> every position's front / back box and SAH cost ->
//      first strict minimum in (axis, position) order -> stable partition of the other two axes by the side flag.
//      Segments of at most max(kSmall, max_tris) triangles are finished by one thread each with the host's sequential
//      sweep, numbering their nodes in pre-order;
//   4. pre-order numbering of the upper tree from subtree sizes (host, a few nodes per kSmall triangles), then every
//      node record is written in the masked 9-float layout and copied back with `order` (= the final x-sorted indices).
// The call owns its stream and device memory (stream-ordered, so a live context on the same device is not synchronised)
// and frees both before it returns.
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>

#include <chrono>
#include <string>
#include <vector>

#include "../../include/fspt_b200.h"
#include "bvh_sah.h"

namespace fspt {
extern thread_local std::string g_create_error;
}

namespace {

constexpr int kThreads = 256;
constexpr int kItems = 8;
constexpr int kChunk = kThreads * kItems;  // positions per block: radix tile, scan tile and level-path chunk
constexpr int kSmall = 64;                 // segments up to this size are finished by one thread
constexpr int kMaxSplitDepth = 4000;       // bvh.js recursion that the host builder refuses to follow
constexpr unsigned kFull = 0xffffffffu;

struct Seg { int32_t lo, hi, node, depth; };
struct Chunk { int32_t seg, c0, c1; };
struct BigNode { float box[6]; int32_t left, right, fin; };  // fin >= 0: this node is the root of finished segment `fin`
struct FinNode { float box[6]; int32_t left, right, lo; };   // left < 0: leaf over [lo, lo + n)
struct Counters { int32_t n_next, n_fin, n_big, depth, fail, n_chunks; };
struct Best { double cost; int32_t axis, pos; };

__device__ __forceinline__ Aabb empty_box() { Aabb b; b.reset(); return b; }

__device__ __forceinline__ Aabb shfl_up(const Aabb& b, int d) {
  Aabb r;
  for (int k = 0; k < 3; ++k) { r.mn[k] = __shfl_up_sync(kFull, b.mn[k], d); r.mx[k] = __shfl_up_sync(kFull, b.mx[k], d); }
  return r;
}
__device__ __forceinline__ Aabb shfl_idx(const Aabb& b, int l) {
  Aabb r;
  for (int k = 0; k < 3; ++k) { r.mn[k] = __shfl_sync(kFull, b.mn[k], l); r.mx[k] = __shfl_sync(kFull, b.mx[k], l); }
  return r;
}
__device__ __forceinline__ Aabb warp_incl(Aabb v) {
  const int lane = threadIdx.x & 31;
  for (int d = 1; d < 32; d <<= 1) { Aabb o = shfl_up(v, d); if (lane >= d) v.grow(o); }
  return v;
}
// union of the aggregates of all earlier threads of the block (thread order = element order)
__device__ Aabb block_excl(const Aabb& agg, Aabb* wsm) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const Aabb incl = warp_incl(agg);
  if (lane == 31) wsm[w] = incl;
  __syncthreads();
  Aabb r = shfl_up(incl, 1);
  if (lane == 0) r.reset();
  for (int j = 0; j < w; ++j) r.grow(wsm[j]);
  __syncthreads();
  return r;
}
__device__ int32_t block_excl_int(int32_t v, int32_t* wsm) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  int32_t incl = v;
  for (int d = 1; d < 32; d <<= 1) { int32_t o = __shfl_up_sync(kFull, incl, d); if (lane >= d) incl += o; }
  if (lane == 31) wsm[w] = incl;
  __syncthreads();
  int32_t r = incl - v;
  for (int j = 0; j < w; ++j) r += wsm[j];
  __syncthreads();
  return r;
}
__device__ __forceinline__ bool better(const Best& b, const Best& a) {  // b precedes a: lower cost, then (axis, position)
  return b.cost < a.cost || (b.cost == a.cost && (b.axis < a.axis || (b.axis == a.axis && b.pos < a.pos)));
}

// ---- 1. boxes, centroid keys ----------------------------------------------------------------------------------------

__device__ __forceinline__ uint64_t order_key(double c) {
  if (c == 0) c = 0.0;  // -0.0 and +0.0 tie under `<`
  const uint64_t u = (uint64_t)__double_as_longlong(c);
  return (u >> 63) ? ~u : (u | 0x8000000000000000ull);
}

__global__ void k_boxes(const double* verts, const double* box_verts, int32_t T, Aabb* tb, Aabb* nb, uint64_t* keys,
                        int32_t* vals, int32_t* bad) {
  const int32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= T) return;
  const double* bv = box_verts ? box_verts : verts;
  Aabb b; b.reset();
  bool ok = true;
  for (int v = 0; v < 3; ++v)
    for (int k = 0; k < 3; ++k) {
      const double x = bv[(size_t)i * 9 + v * 3 + k];
      ok &= finite_coord(x);
      b.add_point(x, k);
    }
  tb[i] = b;
  for (int k = 0; k < 3; ++k) { keys[(size_t)k * T + i] = order_key(b.centroid(k)); vals[(size_t)k * T + i] = i; }
  if (box_verts) {
    Aabb n; n.reset();
    for (int v = 0; v < 3; ++v)
      for (int k = 0; k < 3; ++k) {
        const double x = verts[(size_t)i * 9 + v * 3 + k];
        ok &= finite_coord(x);
        n.add_point(x, k);
      }
    nb[i] = n;
  }
  if (!ok) atomicOr(bad, 1);
}

// ---- exclusive scan of unsigned counts, gridDim.y independent rows of `len` ------------------------------------------

__global__ void k_scan_tiles(uint32_t* data, int32_t len, uint32_t* partial) {
  __shared__ int32_t wsm[kThreads / 32];
  uint32_t* row = data + (size_t)blockIdx.y * len;
  const int32_t base = blockIdx.x * kChunk + threadIdx.x * kItems;
  uint32_t v[kItems], sum = 0;
  for (int j = 0; j < kItems; ++j) { v[j] = base + j < len ? row[base + j] : 0; sum += v[j]; }
  uint32_t run = (uint32_t)block_excl_int((int32_t)sum, wsm);
  for (int j = 0; j < kItems; ++j) if (base + j < len) { row[base + j] = run; run += v[j]; }
  if (threadIdx.x == kThreads - 1) partial[(size_t)blockIdx.y * gridDim.x + blockIdx.x] = run;
}
__global__ void k_scan_partials(uint32_t* partial, int32_t n, int32_t* total) {
  __shared__ int32_t wsm[kThreads / 32];
  __shared__ uint32_t tile_total;
  uint32_t* row = partial + (size_t)blockIdx.x * n;
  uint32_t carry = 0;
  for (int32_t b = 0; b < n; b += kThreads) {
    const int32_t i = b + threadIdx.x;
    const uint32_t v = i < n ? row[i] : 0;
    const uint32_t e = (uint32_t)block_excl_int((int32_t)v, wsm);
    if (i < n) row[i] = carry + e;
    if (threadIdx.x == kThreads - 1) tile_total = e + v;
    __syncthreads();
    carry += tile_total;
    __syncthreads();
  }
  if (total && threadIdx.x == 0) *total = (int32_t)carry;
}
__global__ void k_scan_add(uint32_t* data, int32_t len, const uint32_t* partial) {
  uint32_t* row = data + (size_t)blockIdx.y * len;
  const uint32_t add = partial[(size_t)blockIdx.y * gridDim.x + blockIdx.x];
  const int32_t base = blockIdx.x * kChunk + threadIdx.x * kItems;
  for (int j = 0; j < kItems; ++j) if (base + j < len) row[base + j] += add;
}

// ---- 2. stable LSD radix sort of the three key rows, 8 bits per pass ------------------------------------------------

__global__ void k_radix_hist(const uint64_t* keys, int32_t T, int shift, uint32_t* hist) {
  __shared__ uint32_t h[256];
  const int a = blockIdx.y, tile = blockIdx.x, ntiles = gridDim.x;
  h[threadIdx.x] = 0;
  __syncthreads();
  const uint64_t* kin = keys + (size_t)a * T;
  for (int r = 0; r < kItems; ++r) {
    const int32_t p = tile * kChunk + r * kThreads + threadIdx.x;
    if (p < T) atomicAdd(&h[(kin[p] >> shift) & 255], 1u);
  }
  __syncthreads();
  hist[(size_t)a * 256 * ntiles + (size_t)threadIdx.x * ntiles + tile] = h[threadIdx.x];
}

__global__ void k_radix_scatter(const uint64_t* kin_all, const int32_t* vin_all, uint64_t* kout_all, int32_t* vout_all,
                                int32_t T, int shift, const uint32_t* offs) {
  __shared__ uint32_t base_d[256];
  __shared__ uint32_t wcnt[kThreads / 32][256];
  const int a = blockIdx.y, tile = blockIdx.x, ntiles = gridDim.x;
  const int t = threadIdx.x, lane = t & 31, w = t >> 5;
  const uint64_t* kin = kin_all + (size_t)a * T;
  const int32_t* vin = vin_all + (size_t)a * T;
  uint64_t* kout = kout_all + (size_t)a * T;
  int32_t* vout = vout_all + (size_t)a * T;
  base_d[t] = offs[(size_t)a * 256 * ntiles + (size_t)t * ntiles + tile];
  const unsigned lt = (1u << lane) - 1;
  for (int r = 0; r < kItems; ++r) {
    const int32_t p = tile * kChunk + r * kThreads + t;
    const bool valid = p < T;
    const uint64_t key = valid ? kin[p] : 0;
    const int d = valid ? (int)((key >> shift) & 255) : 256;
    for (int i = t; i < (kThreads / 32) * 256; i += kThreads) (&wcnt[0][0])[i] = 0;
    __syncthreads();
    const unsigned peers = __match_any_sync(kFull, d);
    const int rank = __popc(peers & lt);
    if (valid && rank == 0) wcnt[w][d] = __popc(peers);
    __syncthreads();
    uint32_t run = base_d[t];  // thread t owns digit t: running position of the digit, warp by warp
    for (int j = 0; j < kThreads / 32; ++j) { const uint32_t c = wcnt[j][t]; wcnt[j][t] = run; run += c; }
    base_d[t] = run;
    __syncthreads();
    if (valid) {
      const uint32_t pos = wcnt[w][d] + rank;
      kout[pos] = key;
      vout[pos] = vin[p];
    }
    __syncthreads();
  }
}

// ---- 3. one level of the top-down build ------------------------------------------------------------------------------

struct Level {
  const Seg* seg; int32_t n_seg;
  uint32_t* seg_c0;  // first chunk of each segment
  Chunk* chunks; const int32_t* n_chunks;
  int32_t* seg_axis; int32_t* seg_mid; double* seg_parent; Aabb* seg_box;
  Aabb* cbox;       // [4][cap]: per axis union of tb, [3] = union of nb over axis 0
  Aabb* pre; Aabb* suf;  // [3][cap]
  double* ccost; int32_t* cpos;  // [3][cap]
  int32_t* cnt;     // [3][cap]
  int32_t cap;
};

__device__ __forceinline__ int32_t n_chunks_of(const Seg& s) { return (s.hi - s.lo + kChunk - 1) / kChunk; }

__global__ void k_seg_nchunks(Level L) {
  const int32_t s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s < L.n_seg) L.seg_c0[s] = (uint32_t)n_chunks_of(L.seg[s]);
}
__global__ void k_expand_chunks(Level L) {
  const int32_t s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= L.n_seg) return;
  const Seg g = L.seg[s];
  const int32_t c0 = (int32_t)L.seg_c0[s], n = n_chunks_of(g);
  for (int32_t j = 0; j < n; ++j)
    L.chunks[c0 + j] = Chunk{s, g.lo + j * kChunk, min(g.hi, g.lo + (j + 1) * kChunk)};
}

__global__ void k_chunk_union(Level L, int32_t* const* idx, const Aabb* tb, const Aabb* nb) {
  __shared__ Aabb wsm[kThreads / 32];
  const int32_t c = blockIdx.x;
  if (c >= *L.n_chunks) return;
  const int a = blockIdx.y;
  const Chunk ch = L.chunks[c];
  const int32_t* ix = idx[a < 3 ? a : 0];
  const Aabb* box = a < 3 ? tb : nb;
  Aabb agg; agg.reset();
  for (int j = 0; j < kItems; ++j) {
    const int32_t p = ch.c0 + threadIdx.x * kItems + j;
    if (p < ch.c1) agg.grow(box[ix[p]]);
  }
  Aabb r = block_excl(agg, wsm);
  r.grow(agg);
  if (threadIdx.x == kThreads - 1) L.cbox[(size_t)a * L.cap + c] = r;
}

// one warp per segment: node box, parent area, exclusive prefix / suffix unions over the segment's chunks
__global__ void k_seg_prefix(Level L) {
  const int32_t s = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (s >= L.n_seg) return;
  const int32_t c0 = (int32_t)L.seg_c0[s], n = n_chunks_of(L.seg[s]);
  Aabb box; box.reset();
  for (int32_t j = lane; j < n; j += 32) box.grow(L.cbox[(size_t)3 * L.cap + c0 + j]);
  box = shfl_idx(warp_incl(box), 31);
  if (lane == 0) { L.seg_box[s] = box; L.seg_parent[s] = box.area(); }
  for (int a = 0; a < 3; ++a) {
    const Aabb* cb = L.cbox + (size_t)a * L.cap + c0;
    Aabb carry; carry.reset();
    for (int32_t b = 0; b < n; b += 32) {  // front: chunks before
      const int32_t j = b + lane;
      const Aabb incl = warp_incl(j < n ? cb[j] : empty_box());
      Aabb ex = shfl_up(incl, 1);
      if (lane == 0) ex.reset();
      ex.grow(carry);
      if (j < n) L.pre[(size_t)a * L.cap + c0 + j] = ex;
      carry.grow(shfl_idx(incl, 31));
    }
    carry.reset();
    for (int32_t b = 0; b < n; b += 32) {  // back: chunks after
      const int32_t j = n - 1 - (b + lane);
      const Aabb incl = warp_incl(j >= 0 ? cb[j] : empty_box());
      Aabb ex = shfl_up(incl, 1);
      if (lane == 0) ex.reset();
      ex.grow(carry);
      if (j >= 0) L.suf[(size_t)a * L.cap + c0 + j] = ex;
      carry.grow(shfl_idx(incl, 31));
    }
  }
}

// the SAH cost of every position of a chunk on one axis; the chunk's first strict minimum
__global__ void k_chunk_sweep(Level L, int32_t* const* idx, const Aabb* tb) {
  __shared__ Aabb wsm[kThreads / 32];
  __shared__ double sback[kChunk];
  __shared__ Best bsm[kThreads / 32];
  const int32_t c = blockIdx.x;
  if (c >= *L.n_chunks) return;
  const int a = blockIdx.y;
  const Chunk ch = L.chunks[c];
  const Seg g = L.seg[ch.seg];
  const int32_t n = g.hi - g.lo;
  const double parent = L.seg_parent[ch.seg];
  const int32_t* ix = idx[a];
  // back boxes: element e of the block is position c1 - 1 - e
  Aabb agg; agg.reset();
  for (int j = 0; j < kItems; ++j) {
    const int32_t p = ch.c1 - 1 - (threadIdx.x * kItems + j);
    if (p >= ch.c0) agg.grow(tb[ix[p]]);
  }
  Aabb run = block_excl(agg, wsm);
  run.grow(L.suf[(size_t)a * L.cap + c]);
  for (int j = 0; j < kItems; ++j) {
    const int32_t p = ch.c1 - 1 - (threadIdx.x * kItems + j);
    if (p >= ch.c0) { run.grow(tb[ix[p]]); sback[p - ch.c0] = run.area(); }
  }
  __syncthreads();
  // front boxes and costs: element e is position c0 + e
  agg.reset();
  for (int j = 0; j < kItems; ++j) {
    const int32_t p = ch.c0 + threadIdx.x * kItems + j;
    if (p < ch.c1) agg.grow(tb[ix[p]]);
  }
  run = block_excl(agg, wsm);
  run.grow(L.pre[(size_t)a * L.cap + c]);
  Best b{INFINITY, a, -1};
  for (int j = 0; j < kItems; ++j) {
    const int32_t p = ch.c0 + threadIdx.x * kItems + j;
    if (p < ch.c1) {
      run.grow(tb[ix[p]]);
      const double cost = sah_cost(run.area(), sback[p - ch.c0], parent, p - g.lo, n);
      if (cost < b.cost) { b.cost = cost; b.pos = p; }
    }
  }
  for (int d = 16; d > 0; d >>= 1) {
    Best o{__shfl_down_sync(kFull, b.cost, d), a, __shfl_down_sync(kFull, b.pos, d)};
    if (better(o, b)) b = o;
  }
  if ((threadIdx.x & 31) == 0) bsm[threadIdx.x >> 5] = b;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int j = 1; j < kThreads / 32; ++j) if (better(bsm[j], b)) b = bsm[j];
    L.ccost[(size_t)a * L.cap + c] = b.cost;
    L.cpos[(size_t)a * L.cap + c] = b.pos;
  }
}

// one warp per segment: the split (first strict minimum over axes and chunks), the node record, the two children
__global__ void k_seg_split(Level L, BigNode* big, Seg* next, Seg* fin, Counters* cnt, int32_t small) {
  const int32_t s = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (s >= L.n_seg) return;
  const Seg g = L.seg[s];
  const int32_t c0 = (int32_t)L.seg_c0[s], nc = n_chunks_of(g), n = g.hi - g.lo;
  Best b{INFINITY, 3, -1};
  for (int a = 0; a < 3; ++a)
    for (int32_t j = lane; j < nc; j += 32) {
      const Best o{L.ccost[(size_t)a * L.cap + c0 + j], a, L.cpos[(size_t)a * L.cap + c0 + j]};
      if (o.pos >= 0 && better(o, b)) b = o;
    }
  for (int d = 16; d > 0; d >>= 1) {
    Best o{__shfl_down_sync(kFull, b.cost, d), __shfl_down_sync(kFull, b.axis, d), __shfl_down_sync(kFull, b.pos, d)};
    if (better(o, b)) b = o;
  }
  if (lane != 0) return;
  const Aabb box = L.seg_box[s];
  BigNode& nd = big[g.node];
  for (int k = 0; k < 3; ++k) { nd.box[k] = __double2float_rn(box.mn[k]); nd.box[3 + k] = __double2float_rn(box.mx[k]); }
  nd.fin = -1;
  const int32_t best_i = b.pos < 0 ? -1 : b.pos - g.lo + 1;
  if (b.pos < 0 || best_i >= n || g.depth > kMaxSplitDepth) {  // JS: TypeError on an undefined axis / unbounded recursion
    atomicOr(&cnt->fail, 1);
    L.seg_axis[s] = -1;
    nd.left = nd.right = -1;
    return;
  }
  const int32_t mid = g.lo + best_i;
  L.seg_axis[s] = b.axis;
  L.seg_mid[s] = mid;
  const int32_t id = atomicAdd(&cnt->n_big, 2);
  nd.left = id; nd.right = id + 1;
  atomicMax(&cnt->depth, g.depth + 1);
  const Seg kids[2] = {{g.lo, mid, id, g.depth + 1}, {mid, g.hi, id + 1, g.depth + 1}};
  for (const Seg& k : kids) {
    BigNode& kn = big[k.node];
    if (k.hi - k.lo <= small) {
      const int32_t f = atomicAdd(&cnt->n_fin, 1);
      fin[f] = k;
      kn.fin = f;
    } else {
      next[atomicAdd(&cnt->n_next, 1)] = k;
      kn.fin = -1;
    }
  }
}

__global__ void k_mark_side(Level L, int32_t* const* idx, uint8_t* side) {
  const int32_t c = blockIdx.x;
  if (c >= *L.n_chunks) return;
  const Chunk ch = L.chunks[c];
  const int axis = L.seg_axis[ch.seg];
  if (axis < 0) return;
  const int32_t mid = L.seg_mid[ch.seg];
  for (int32_t p = ch.c0 + threadIdx.x; p < ch.c1; p += kThreads) side[idx[axis][p]] = p < mid;
}

__global__ void k_part_count(Level L, int32_t* const* idx, const uint8_t* side) {
  __shared__ int32_t wsm[kThreads / 32];
  const int32_t c = blockIdx.x;
  if (c >= *L.n_chunks) return;
  const int a = blockIdx.y;
  const Chunk ch = L.chunks[c];
  const int axis = L.seg_axis[ch.seg];
  if (axis < 0 || axis == a) return;
  int32_t k = 0;
  for (int32_t p = ch.c0 + threadIdx.x; p < ch.c1; p += kThreads) k += side[idx[a][p]];
  const int32_t e = block_excl_int(k, wsm);
  if (threadIdx.x == kThreads - 1) L.cnt[(size_t)a * L.cap + c] = e + k;
}

// one warp per segment: left-goers of the earlier chunks of the segment, per partitioned axis
__global__ void k_seg_offsets(Level L) {
  const int32_t s = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (s >= L.n_seg) return;
  const int axis = L.seg_axis[s];
  if (axis < 0) return;
  const int32_t c0 = (int32_t)L.seg_c0[s], n = n_chunks_of(L.seg[s]);
  for (int a = 0; a < 3; ++a) {
    if (a == axis) continue;
    int32_t* cn = L.cnt + (size_t)a * L.cap + c0;
    int32_t carry = 0;
    for (int32_t b = 0; b < n; b += 32) {
      const int32_t j = b + lane;
      const int32_t v = j < n ? cn[j] : 0;
      int32_t incl = v;
      for (int d = 1; d < 32; d <<= 1) { const int32_t o = __shfl_up_sync(kFull, incl, d); if (lane >= d) incl += o; }
      if (j < n) cn[j] = carry + incl - v;
      carry += __shfl_sync(kFull, incl, 31);
    }
  }
}

// _constructCachedIndexList (bvh.js:52-76): stable partition of the two other axes into tmp, by position
__global__ void k_part_scatter(Level L, int32_t* const* idx, int32_t* const* tmp, const uint8_t* side) {
  __shared__ int32_t wsm[kThreads / 32];
  const int32_t c = blockIdx.x;
  if (c >= *L.n_chunks) return;
  const int a = blockIdx.y;
  const Chunk ch = L.chunks[c];
  const int axis = L.seg_axis[ch.seg];
  if (axis < 0 || axis == a) return;
  const Seg g = L.seg[ch.seg];
  const int32_t mid = L.seg_mid[ch.seg], left_before = L.cnt[(size_t)a * L.cap + c];
  const int32_t* ix = idx[a];
  int32_t v[kItems];
  uint8_t f[kItems];
  int32_t k = 0;
  for (int j = 0; j < kItems; ++j) {
    const int32_t p = ch.c0 + threadIdx.x * kItems + j;
    v[j] = p < ch.c1 ? ix[p] : -1;
    f[j] = v[j] >= 0 ? side[v[j]] : 0;
    k += f[j];
  }
  int32_t l = block_excl_int(k, wsm);  // left-goers of the chunk before this thread's items
  for (int j = 0; j < kItems; ++j) {
    const int32_t e = threadIdx.x * kItems + j;  // element within the chunk
    if (v[j] < 0) break;
    const int32_t dst = f[j] ? g.lo + left_before + l : mid + (ch.c0 - g.lo - left_before) + (e - l);
    tmp[a][dst] = v[j];
    l += f[j];
  }
}

__global__ void k_copy_back(Level L, int32_t* const* idx, int32_t* const* tmp) {
  const int32_t c = blockIdx.x;
  if (c >= *L.n_chunks) return;
  const int a = blockIdx.y;
  const Chunk ch = L.chunks[c];
  const int axis = L.seg_axis[ch.seg];
  if (axis < 0 || axis == a) return;
  for (int32_t p = ch.c0 + threadIdx.x; p < ch.c1; p += kThreads) idx[a][p] = tmp[a][p];
}

// ---- small segments: the host builder's sequential recursion, one thread per segment, nodes in pre-order -----------

__global__ void k_finish(const Seg* fin, int32_t n_fin, int32_t* const* idx, int32_t* const* tmp, const Aabb* tb,
                         const Aabb* nb, double* sback, uint8_t* side, FinNode* fnodes, int32_t* fcount, Counters* cnt,
                         int32_t max_tris) {
  const int32_t f = blockIdx.x * blockDim.x + threadIdx.x;
  if (f >= n_fin) return;
  const Seg s = fin[f];
  FinNode* out = fnodes + 2 * (size_t)s.lo;  // a subtree over n triangles has at most 2n - 1 nodes
  struct Item { int32_t lo, hi, depth, parent, which; };
  Item st[kSmall + 2];
  int sp = 0, count = 0, maxd = s.depth;
  st[sp++] = Item{s.lo, s.hi, s.depth, -1, 0};
  while (sp > 0) {
    const Item it = st[--sp];
    const int32_t self = count++;
    if (it.parent >= 0) { if (it.which) out[it.parent].right = self; else out[it.parent].left = self; }
    maxd = max(maxd, it.depth);
    const int32_t lo = it.lo, hi = it.hi, n = hi - lo;
    Aabb box; box.reset();
    for (int32_t i = lo; i < hi; ++i) box.grow(nb[idx[0][i]]);  // BoundingBox.addNode, bvh.js:122-128
    FinNode& nd = out[self];
    for (int k = 0; k < 3; ++k) { nd.box[k] = __double2float_rn(box.mn[k]); nd.box[3 + k] = __double2float_rn(box.mx[k]); }
    nd.left = nd.right = -1;
    nd.lo = lo;
    if (n <= max_tris) continue;  // bvh.js:22
    const double parent = box.area();
    double best = INFINITY;
    int best_axis = -1;
    int32_t best_i = -1;
    for (int axis = 0; axis < 3; ++axis) {  // Node.setSplit, bvh.js:168-197
      const int32_t* ix = idx[axis];
      Aabb bb; bb.reset();
      for (int32_t i = hi - 1; i >= lo; --i) { bb.grow(tb[ix[i]]); sback[i] = bb.area(); }
      bb.reset();
      for (int32_t i = lo; i < hi; ++i) {
        bb.grow(tb[ix[i]]);
        const double cost = sah_cost(bb.area(), sback[i], parent, i - lo, n);
        if (cost < best) { best = cost; best_i = i - lo + 1; best_axis = axis; }
      }
    }
    if (best_axis < 0 || best_i >= n || it.depth > kMaxSplitDepth) { atomicOr(&cnt->fail, 1); break; }
    const int32_t mid = lo + best_i;
    for (int32_t i = lo; i < hi; ++i) side[idx[best_axis][i]] = i < mid;
    for (int which = 0; which < 2; ++which) {
      const int axis = (best_axis + 1 + which) % 3;
      int32_t* ix = idx[axis];
      int32_t* t = tmp[which];
      int32_t l = lo, r = 0;
      for (int32_t i = lo; i < hi; ++i) { const int32_t v = ix[i]; if (side[v]) ix[l++] = v; else t[lo + r++] = v; }
      for (int32_t i = 0; i < r; ++i) ix[l + i] = t[lo + i];
    }
    st[sp++] = Item{mid, hi, it.depth + 1, self, 1};  // right below left: the left subtree is numbered first
    st[sp++] = Item{lo, mid, it.depth + 1, self, 0};
  }
  fcount[f] = count;
  atomicMax(&cnt->depth, maxd);
}

// ---- 4. the masked bvhBuffer records (main.js:272-282, 366-392) ------------------------------------------------------

__device__ __forceinline__ void put_node(float* out, int32_t at, int32_t l, int32_t r, int32_t t, const float* box) {
  float* p = out + (size_t)at * 9;
  p[0] = __int_as_float(l); p[1] = __int_as_float(r); p[2] = __int_as_float(t);
  for (int k = 0; k < 6; ++k) p[3 + k] = box[k];
}
__global__ void k_emit_big(const BigNode* big, int32_t n_big, const int32_t* pre, float* out) {
  const int32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_big || big[i].fin >= 0) return;
  put_node(out, pre[i], pre[big[i].left], pre[big[i].right], -1, big[i].box);
}
__global__ void k_emit_fin(const Seg* fin, int32_t n_fin, const FinNode* fnodes, const int32_t* fcount, const int32_t* pre,
                           float* out) {
  const int32_t f = blockIdx.x * blockDim.x + threadIdx.x;
  if (f >= n_fin) return;
  const Seg s = fin[f];
  const int32_t base = pre[s.node];
  const FinNode* nd = fnodes + 2 * (size_t)s.lo;
  for (int32_t j = 0; j < fcount[f]; ++j) {
    if (nd[j].left < 0) put_node(out, base + j, 0, 0, nd[j].lo, nd[j].box);  // leaf: triangle index = its first position
    else put_node(out, base + j, base + nd[j].left, base + nd[j].right, -1, nd[j].box);
  }
}

// ---- host side --------------------------------------------------------------------------------------------------------

int fail(int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  fspt::g_create_error = buf;
  return code;
}

// The stream and every device block of one call; released (stream-ordered) when the call returns.
struct Scope {
  int prev_device = -1;
  cudaStream_t stream = nullptr;
  std::vector<void*> blocks;
  ~Scope() {
    for (void* p : blocks) cudaFreeAsync(p, stream);
    if (stream) { cudaStreamSynchronize(stream); cudaStreamDestroy(stream); }
    if (prev_device >= 0) cudaSetDevice(prev_device);
  }
  template <class T>
  cudaError_t alloc(T** p, size_t count) {
    void* q = nullptr;
    const cudaError_t e = cudaMallocAsync(&q, (count > 0 ? count : 1) * sizeof(T), stream);
    if (e == cudaSuccess) blocks.push_back(q);
    *p = static_cast<T*>(q);
    return e;
  }
};

#define CKD(call)                                                                                  \
  do {                                                                                             \
    const cudaError_t e_ = (call);                                                                 \
    if (e_ != cudaSuccess) return fail(FSPT_E_CUDA, "fspt_bvh_build_device: %s failed: %s", #call, \
                                       cudaGetErrorString(e_));                                    \
  } while (0)

int grid_of(int64_t n, int per_block) { return (int)((n + per_block - 1) / per_block); }

// exclusive scan of `rows` rows of `len` counts in place; *total (if given) receives the total of row 0
int scan_rows(uint32_t* data, int32_t len, int rows, uint32_t* partial, int32_t* total, cudaStream_t st) {
  const int nb = grid_of(len, kChunk);
  k_scan_tiles<<<dim3(nb, rows), kThreads, 0, st>>>(data, len, partial);
  k_scan_partials<<<rows, kThreads, 0, st>>>(partial, nb, total);
  k_scan_add<<<dim3(nb, rows), kThreads, 0, st>>>(data, len, partial);
  CKD(cudaGetLastError());
  return FSPT_OK;
}

int build_device(Scope& sc, const double* verts, const double* box_verts, int32_t T, int32_t max_tris, float* nodes_out,
                 int32_t* order_out, int32_t* n_nodes_out, int32_t* depth_out) {
  cudaStream_t st = sc.stream;
  const bool timing = getenv("FSPT_TIMING") != nullptr;
  auto t_prev = std::chrono::steady_clock::now();
  auto lap = [&](const char* what) -> int {
    if (!timing) return FSPT_OK;
    CKD(cudaStreamSynchronize(st));
    const auto now = std::chrono::steady_clock::now();
    fprintf(stderr, "[fspt bvh device] %-24s %8.1f ms\n", what, std::chrono::duration<double, std::milli>(now - t_prev).count());
    t_prev = now;
    return FSPT_OK;
  };
  const size_t n = (size_t)T;
  const int32_t small = kSmall > max_tris ? kSmall : max_tris;
  double *d_verts, *d_box_verts = nullptr;
  Aabb *tb, *nb;
  uint64_t* keys;  // [2][3][T]; the second half is reused as the finisher's sback (doubles)
  int32_t* vals;   // [2][3][T]; after the sort [0] holds idx[3], [1] is partition scratch
  int32_t* bad;
  uint8_t* side;
  Counters* cnt;
  CKD(sc.alloc(&d_verts, n * 9));
  if (box_verts) CKD(sc.alloc(&d_box_verts, n * 9));
  CKD(sc.alloc(&tb, n));
  if (box_verts) CKD(sc.alloc(&nb, n)); else nb = tb;
  CKD(sc.alloc(&keys, 6 * n));
  CKD(sc.alloc(&vals, 6 * n));
  CKD(sc.alloc(&bad, 1));
  CKD(sc.alloc(&side, n));
  CKD(sc.alloc(&cnt, 1));
  CKD(cudaMemcpyAsync(d_verts, verts, n * 9 * sizeof(double), cudaMemcpyHostToDevice, st));
  if (box_verts) CKD(cudaMemcpyAsync(d_box_verts, box_verts, n * 9 * sizeof(double), cudaMemcpyHostToDevice, st));
  CKD(cudaMemsetAsync(bad, 0, sizeof(int32_t), st));
  if (int rc = lap("upload")) return rc;
  k_boxes<<<grid_of(T, kThreads), kThreads, 0, st>>>(d_verts, d_box_verts, T, tb, box_verts ? nb : nullptr, keys, vals, bad);
  CKD(cudaGetLastError());
  int32_t h_bad = 0;
  CKD(cudaMemcpyAsync(&h_bad, bad, sizeof h_bad, cudaMemcpyDeviceToHost, st));
  CKD(cudaStreamSynchronize(st));
  if (h_bad) return fail(FSPT_E_INVALID, "fspt_bvh_build_device: a vertex coordinate is NaN or infinite");
  if (int rc = lap("boxes + centroids")) return rc;

  {  // _sortIndices x3 (bvh.js:78-90)
    const int ntiles = grid_of(T, kChunk);
    uint32_t *hist, *partial;
    CKD(sc.alloc(&hist, (size_t)3 * 256 * ntiles));
    CKD(sc.alloc(&partial, (size_t)3 * grid_of((int64_t)256 * ntiles, kChunk)));
    for (int pass = 0; pass < 8; ++pass) {
      const int src = pass & 1;
      k_radix_hist<<<dim3(ntiles, 3), 256, 0, st>>>(keys + src * 3 * n, T, pass * 8, hist);
      if (int rc = scan_rows(hist, 256 * ntiles, 3, partial, nullptr, st)) return rc;
      k_radix_scatter<<<dim3(ntiles, 3), kThreads, 0, st>>>(keys + src * 3 * n, vals + src * 3 * n, keys + (1 - src) * 3 * n,
                                                           vals + (1 - src) * 3 * n, T, pass * 8, hist);
      CKD(cudaGetLastError());
    }
  }
  if (int rc = lap("presort x3")) return rc;

  // position-indexed index rows: idx[0..2] (the sorted rows, partitioned in place) and tmp[0..2] (partition scratch)
  int32_t** idx;
  CKD(sc.alloc(&idx, 6));
  {
    int32_t* rows[6];
    for (int r = 0; r < 6; ++r) rows[r] = vals + r * n;
    CKD(cudaMemcpyAsync(idx, rows, sizeof rows, cudaMemcpyHostToDevice, st));
  }
  int32_t** tmp = idx + 3;
  // upper tree: segments of more than `small` triangles, one level at a time
  const int32_t cap_seg = T / (small + 1) + 2;              // disjoint segments of > small triangles, per level
  const int32_t cap_chunk = grid_of(T, kChunk) + cap_seg;  // chunks of one level
  const int32_t cap_big = 2 * T + 1;
  Seg *seg_a, *seg_b, *fin;
  BigNode* big;
  Level L{};
  L.cap = cap_chunk;
  CKD(sc.alloc(&seg_a, cap_seg));
  CKD(sc.alloc(&seg_b, cap_seg));
  CKD(sc.alloc(&fin, n));
  CKD(sc.alloc(&big, cap_big));
  CKD(sc.alloc(&L.seg_c0, cap_seg));
  uint32_t* seg_partial;
  CKD(sc.alloc(&seg_partial, grid_of(cap_seg, kChunk)));
  CKD(sc.alloc(&L.chunks, cap_chunk));
  CKD(sc.alloc(&L.seg_axis, cap_seg));
  CKD(sc.alloc(&L.seg_mid, cap_seg));
  CKD(sc.alloc(&L.seg_parent, cap_seg));
  CKD(sc.alloc(&L.seg_box, cap_seg));
  CKD(sc.alloc(&L.cbox, (size_t)4 * cap_chunk));
  CKD(sc.alloc(&L.pre, (size_t)3 * cap_chunk));
  CKD(sc.alloc(&L.suf, (size_t)3 * cap_chunk));
  CKD(sc.alloc(&L.ccost, (size_t)3 * cap_chunk));
  CKD(sc.alloc(&L.cpos, (size_t)3 * cap_chunk));
  CKD(sc.alloc(&L.cnt, (size_t)3 * cap_chunk));
  int32_t* d_nchunks = &cnt->n_chunks;
  L.n_chunks = d_nchunks;

  Counters h{};
  h.n_big = 1;
  const Seg root{0, T, 0, 0};
  int32_t n_seg = 0;
  if (T <= small) {
    h.n_fin = 1;
    CKD(cudaMemcpyAsync(fin, &root, sizeof root, cudaMemcpyHostToDevice, st));
    const int32_t f0 = 0;
    CKD(cudaMemcpyAsync(&big[0].fin, &f0, sizeof f0, cudaMemcpyHostToDevice, st));
  } else {
    n_seg = 1;
    CKD(cudaMemcpyAsync(seg_a, &root, sizeof root, cudaMemcpyHostToDevice, st));
  }
  CKD(cudaMemcpyAsync(cnt, &h, sizeof h, cudaMemcpyHostToDevice, st));
  Seg *cur = seg_a, *nxt = seg_b;
  int levels = 0;
  while (n_seg > 0) {
    L.seg = cur;
    L.n_seg = n_seg;
    const int chunk_grid = grid_of(T, kChunk) + n_seg;  // bound; blocks past *n_chunks return at once
    const int seg_grid = grid_of(n_seg, kThreads), warp_grid = grid_of((int64_t)n_seg * 32, kThreads);
    k_seg_nchunks<<<seg_grid, kThreads, 0, st>>>(L);
    if (int rc = scan_rows(L.seg_c0, n_seg, 1, seg_partial, d_nchunks, st)) return rc;
    k_expand_chunks<<<seg_grid, kThreads, 0, st>>>(L);
    k_chunk_union<<<dim3(chunk_grid, 4), kThreads, 0, st>>>(L, idx, tb, nb);
    k_seg_prefix<<<warp_grid, kThreads, 0, st>>>(L);
    k_chunk_sweep<<<dim3(chunk_grid, 3), kThreads, 0, st>>>(L, idx, tb);
    k_seg_split<<<warp_grid, kThreads, 0, st>>>(L, big, nxt, fin, cnt, small);
    k_mark_side<<<chunk_grid, kThreads, 0, st>>>(L, idx, side);
    k_part_count<<<dim3(chunk_grid, 3), kThreads, 0, st>>>(L, idx, side);
    k_seg_offsets<<<warp_grid, kThreads, 0, st>>>(L);
    k_part_scatter<<<dim3(chunk_grid, 3), kThreads, 0, st>>>(L, idx, tmp, side);
    k_copy_back<<<dim3(chunk_grid, 3), kThreads, 0, st>>>(L, idx, tmp);
    CKD(cudaGetLastError());
    CKD(cudaMemcpyAsync(&h, cnt, sizeof h, cudaMemcpyDeviceToHost, st));
    CKD(cudaStreamSynchronize(st));
    if (h.fail) return fail(FSPT_E_LIMIT, "fspt_bvh_build_device: no split found (the JavaScript builder would not terminate)");
    n_seg = h.n_next;
    CKD(cudaMemsetAsync(&cnt->n_next, 0, sizeof(int32_t), st));
    Seg* t = cur; cur = nxt; nxt = t;
    ++levels;
  }
  if (int rc = lap("build: upper levels")) return rc;
  FinNode* fnodes;
  int32_t* fcount;
  CKD(sc.alloc(&fnodes, 2 * n));
  CKD(sc.alloc(&fcount, (size_t)h.n_fin));
  k_finish<<<grid_of(h.n_fin, 128), 128, 0, st>>>(fin, h.n_fin, idx, tmp, tb, nb, reinterpret_cast<double*>(keys + 3 * n),
                                                 side, fnodes, fcount, cnt, max_tris);
  CKD(cudaGetLastError());
  CKD(cudaMemcpyAsync(&h, cnt, sizeof h, cudaMemcpyDeviceToHost, st));
  CKD(cudaStreamSynchronize(st));
  if (h.fail) return fail(FSPT_E_LIMIT, "fspt_bvh_build_device: no split found (the JavaScript builder would not terminate)");
  if (int rc = lap("build: small segments")) return rc;

  // serializeTree (bvh.js:33-50) + flatten: pre-order numbers of the upper tree from subtree sizes.  Children are
  // allocated after their parent, so sizes go by descending and numbers by ascending id.
  std::vector<BigNode> hb((size_t)h.n_big);
  std::vector<Seg> hf((size_t)h.n_fin);
  std::vector<int32_t> hc((size_t)h.n_fin), size((size_t)h.n_big), pre((size_t)h.n_big);
  CKD(cudaMemcpyAsync(hb.data(), big, hb.size() * sizeof(BigNode), cudaMemcpyDeviceToHost, st));
  CKD(cudaMemcpyAsync(hc.data(), fcount, hc.size() * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  CKD(cudaStreamSynchronize(st));
  for (int32_t i = h.n_big - 1; i >= 0; --i)
    size[i] = hb[i].fin >= 0 ? hc[hb[i].fin] : 1 + size[hb[i].left] + size[hb[i].right];
  pre[0] = 0;
  for (int32_t i = 0; i < h.n_big; ++i)
    if (hb[i].fin < 0) { pre[hb[i].left] = pre[i] + 1; pre[hb[i].right] = pre[i] + 1 + size[hb[i].left]; }
  const int32_t n_nodes = size[0];
  int32_t* d_pre;
  float* d_out;
  CKD(sc.alloc(&d_pre, pre.size()));
  CKD(sc.alloc(&d_out, (size_t)n_nodes * 9));
  CKD(cudaMemcpyAsync(d_pre, pre.data(), pre.size() * sizeof(int32_t), cudaMemcpyHostToDevice, st));
  k_emit_big<<<grid_of(h.n_big, kThreads), kThreads, 0, st>>>(big, h.n_big, d_pre, d_out);
  k_emit_fin<<<grid_of(h.n_fin, 128), 128, 0, st>>>(fin, h.n_fin, fnodes, fcount, d_pre, d_out);
  CKD(cudaGetLastError());
  CKD(cudaMemcpyAsync(nodes_out, d_out, (size_t)n_nodes * 9 * sizeof(float), cudaMemcpyDeviceToHost, st));
  CKD(cudaMemcpyAsync(order_out, vals, n * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  CKD(cudaStreamSynchronize(st));
  if (int rc = lap("flatten + download")) return rc;
  if (timing) fprintf(stderr, "[fspt bvh device] %d upper levels, %d upper nodes, %d small segments\n", levels, h.n_big, h.n_fin);
  if (n_nodes_out) *n_nodes_out = n_nodes;
  if (depth_out) *depth_out = h.depth;
  return FSPT_OK;
}

}  // namespace

extern "C" int fspt_device_check(int32_t device) {
  int n_dev = 0;
  const cudaError_t e = cudaGetDeviceCount(&n_dev);
  if (e != cudaSuccess || n_dev <= 0) {
    (void)cudaGetLastError();
    return fail(FSPT_E_CUDA, "no CUDA device: %s (this library has no CPU fallback)", cudaGetErrorString(e));
  }
  if (device < 0 || device >= n_dev) return fail(FSPT_E_INVALID, "device %d out of range (%d present)", device, n_dev);
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) != cudaSuccess || prop.major != 10)
    return fail(FSPT_E_CUDA, "device %d is sm_%d%d; kernels are built for sm_100a only (no CPU fallback)", device, prop.major,
                prop.minor);
  return FSPT_OK;
}

extern "C" int fspt_bvh_build_device(int32_t device, const double* verts, const double* box_verts, int32_t n_tris,
                                     int32_t max_tris, float* nodes_out, int32_t* order_out, int32_t* n_nodes_out,
                                     int32_t* depth_out) {
  if (!verts || !nodes_out || !order_out || n_tris <= 0 || max_tris <= 0)
    return fail(FSPT_E_INVALID, "fspt_bvh_build_device: bad arguments");
  if (int rc = fspt_device_check(device)) return rc;
  Scope sc;
  if (cudaGetDevice(&sc.prev_device) != cudaSuccess) sc.prev_device = -1;
  cudaError_t e = cudaSetDevice(device);
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&sc.stream, cudaStreamNonBlocking);
  if (e != cudaSuccess) return fail(FSPT_E_CUDA, "fspt_bvh_build_device: device %d: %s", device, cudaGetErrorString(e));
  return build_device(sc, verts, box_verts, n_tris, max_tris, nodes_out, order_out, n_nodes_out, depth_out);
}
