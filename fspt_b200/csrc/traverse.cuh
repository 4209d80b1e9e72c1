// traverse.cuh -- closest-hit BVH traversal + Moller-Trumbore, persistent warps with dynamic ray fetch.
//
// Replaces intersectScene / rayBoxIntersect / processLeaf / rayTriangleIntersect of the reference
// (tracer.fs:300-326,355-404; counter variant bvh_test.fs:173-221).  Per ray the sequence of visited nodes,
// the pruning comparisons and the triangle-test order are exactly the reference's, so (index, t, count)
// are bit-identical:
//   - near child first, `leftHit > rightHit` sends the ray right (ties go left), far child deferred
//     (tracer.fs:382-392); deferred nodes are NOT re-tested against result.t when popped (tracer.fs:401);
//   - a leaf tests exactly LEAF_SIZE = 4 consecutive triangles starting at its first one, over-reading
//     into the next leaf (tracer.fs:355-364); strict `<` keeps the first hit on ties (tracer.fs:359);
//   - slab test: (b - o) * (1/d), IEEE division, min/max = minNum/maxNum, `tMax >= tMin && tMax > 0`
//     (tracer.fs:317-326); no FMA contraction anywhere (file is compiled with --fmad=false).
// The two box tests the reference also performs on leaf visits (children 0,0 -> root box, tracer.fs:377-378)
// have no observable effect and are skipped.
//
// Execution model: one ray per lane, a warp keeps running until fewer than REFILL lanes still have a ray,
// then the idle lanes are refilled from a global queue (__ballot_sync + popc prefix = the compaction), so
// short rays do not wait for the longest ray of their warp.  Inside the loop the warp votes each iteration
// whether to run an interior step or a leaf step (majority of lanes).
//
// Round-2 changes, each from the ncu source page of the round-1 build (profiles/r01_final_k_trace_ncu.txt):
//   - SHORT STACK IN SHARED MEMORY: the reference's `int stack[64]` lived in local memory, whose L1 hit rate
//     was 71-78 % (it competes with nodes and triangles), so every fourth pop waited for L2 before the dependent
//     node fetch could issue.  The first TRACE_SMEM_STACK entries now sit in shared memory, laid out
//     [depth][thread] (bank = lane for every per-lane depth: conflict-free), deeper entries spill to local memory.
//   - BROADCAST OPERANDS: ray origin / direction / inverse direction are kept as scalars and packed at the use
//     site; ptxas folds `mov.b64 {x, x}` into the `.F32` scalar-broadcast operand of FADD2/FMUL2, which frees the
//     nine registers the materialised (x, x) pairs occupied.
#pragma once
#include "camera.cuh"
#include "device_common.cuh"

struct TraceArgs {
  const float4* nodes;
  const float4* tris;
  cudaTextureObject_t nodes_tex;  // the node array again as a linear texture (second L1 data pipe)
  int root_ref;
  PathState ps;           // rays in, hits out (words 0..2 of the path record)
  const float4* shadow_rays;  // shadow rays, dense, 2 words each: origin | record position, direction | - (written by k_shade)
  const int* counts;      // counts[0] = #continuation, counts[1] = #shadow
  int* next;              // work-fetch cursor (zeroed before launch)
  unsigned long long* stats;  // [0] rays, [1] node visits, [2] leaf visits
  int* count_out;         // per-slot visit count (debug / bvh_test mode) or NULL
  unsigned char* hit_flag;  // per record position: 1 = hit (read coalesced by k_shade) or NULL
  FrameParams f;          // CAMERA mode: primary rays are generated in the fetch instead of being read
  const float* rb_cam;
  int n_samples;
  FastDiv div_s;          // by n_samples
  int anyhit;             // 1: hit-or-miss rays (shadow rays, marked last-bounce rays) stop at their first intersection
  const int* list;        // LIST: the slots of the pixels this wave renders (adaptive.cuh); last, so that the other
                          // instantiations keep their parameter offsets and instructions
};

#ifndef TRACE_THREADS
#define TRACE_THREADS 128
#endif
#ifndef TRACE_REFILL
#define TRACE_REFILL 16      /* a warp fetches new rays when fewer lanes than this still hold one (with 36 warps/SM:
                                16 is 2.3 % faster than 12 on the 82 k-triangle scene, 1.8 % slower on 1 M triangles) */
#endif
#ifndef TRACE_SMEM_STACK
#define TRACE_SMEM_STACK 12  /* stack entries per thread held in shared memory; the rest spill to local memory
                                (0: every entry spills) */
#endif
#ifndef TRACE_MIN_BLOCKS
#define TRACE_MIN_BLOCKS 9   /* resident CTAs per SM the register allocation is held to (9 x 128 threads = 56 registers) */
#endif

__device__ __forceinline__ float slab(float bminx, float bminy, float bminz, float bmaxx, float bmaxy, float bmaxz,
                                      float ox, float oy, float oz, float ix, float iy, float iz) {
  const float t1x = (bminx - ox) * ix, t2x = (bmaxx - ox) * ix;
  const float t1y = (bminy - oy) * iy, t2y = (bmaxy - oy) * iy;
  const float t1z = (bminz - oz) * iz, t2z = (bmaxz - oz) * iz;
  const float tMax = fminf(fminf(fmaxf(t1x, t2x), fmaxf(t1y, t2y)), fmaxf(t1z, t2z));
  const float tMin = fmaxf(fmaxf(fminf(t1x, t2x), fminf(t1y, t2y)), fminf(t1z, t2z));
  return (tMax >= tMin && tMax > 0.0f) ? tMin : FSPT_MAX_T;
}

// Blackwell's packed f32x2 pipe: FADD2 / FMUL2 perform two independent IEEE round-to-nearest f32 operations per
// instruction.  pack2(x, x) of a scalar costs nothing: ptxas folds it into the instruction's `.F32` broadcast operand.
typedef unsigned long long f32x2;
__device__ __forceinline__ f32x2 pack2(float lo, float hi) { f32x2 r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi)); return r; }
__device__ __forceinline__ f32x2 bc2(float v) { return pack2(v, v); }
__device__ __forceinline__ void unpack2(f32x2 v, float& lo, float& hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ f32x2 sub2(f32x2 a, f32x2 b) { f32x2 r; asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ f32x2 add2(f32x2 a, f32x2 b) { f32x2 r; asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ f32x2 mul2(f32x2 a, f32x2 b) { f32x2 r; asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }

// Both child boxes at once (lane 0 of a pair = left child, lane 1 = right child): the 24 subtract/multiply
// operations of the two slab tests issue as 12 instructions.  Bitwise identical to slab().
__device__ __forceinline__ void slab_pair(const float4 w0, const float4 w1, const float4 w2, f32x2 ox2, f32x2 oy2, f32x2 oz2,
                                          f32x2 ix2, f32x2 iy2, f32x2 iz2, float& lh, float& rh) {
  // record words: w0 = (lmin.x rmin.x lmin.y rmin.y)  w1 = (lmin.z rmin.z lmax.x rmax.x)  w2 = (lmax.y rmax.y lmax.z rmax.z)
  const f32x2 t1x = mul2(sub2(pack2(w0.x, w0.y), ox2), ix2), t1y = mul2(sub2(pack2(w0.z, w0.w), oy2), iy2);
  const f32x2 t1z = mul2(sub2(pack2(w1.x, w1.y), oz2), iz2), t2x = mul2(sub2(pack2(w1.z, w1.w), ox2), ix2);
  const f32x2 t2y = mul2(sub2(pack2(w2.x, w2.y), oy2), iy2), t2z = mul2(sub2(pack2(w2.z, w2.w), oz2), iz2);
  float a1x, b1x, a1y, b1y, a1z, b1z, a2x, b2x, a2y, b2y, a2z, b2z;
  unpack2(t1x, a1x, b1x); unpack2(t1y, a1y, b1y); unpack2(t1z, a1z, b1z);
  unpack2(t2x, a2x, b2x); unpack2(t2y, a2y, b2y); unpack2(t2z, a2z, b2z);
  const float lMax = fminf(fminf(fmaxf(a1x, a2x), fmaxf(a1y, a2y)), fmaxf(a1z, a2z));
  const float lMin = fmaxf(fmaxf(fminf(a1x, a2x), fminf(a1y, a2y)), fminf(a1z, a2z));
  const float rMax = fminf(fminf(fmaxf(b1x, b2x), fmaxf(b1y, b2y)), fmaxf(b1z, b2z));
  const float rMin = fmaxf(fmaxf(fminf(b1x, b2x), fminf(b1y, b2y)), fminf(b1z, b2z));
  lh = (lMax >= lMin && lMax > 0.0f) ? lMin : FSPT_MAX_T;
  rh = (rMax >= rMin && rMax > 0.0f) ? rMin : FSPT_MAX_T;
}

// rayTriangleIntersect with e1/e2 precomputed; predicates are the reference's conditions, un-negated, so
// NaN behaves identically (tracer.fs:305,309,312,314)
__device__ __forceinline__ float tri_test(const float4 q0, const float4 q1, const float4 q2, float ox, float oy,
                                          float oz, float dx, float dy, float dz) {
  const float e1x = q0.w, e1y = q1.x, e1z = q1.y, e2x = q1.z, e2y = q1.w, e2z = q2.x;
  const float px = dy * e2z - e2y * dz, py = dz * e2x - e2z * dx, pz = dx * e2y - e2x * dy;  // cross(dir,e2)
  const float det = e1x * px + e1y * py + e1z * pz;
  if (fabsf(det) < FSPT_EPSILON) return FSPT_MAX_T;
  const float invDet = 1.0f / det;
  const float tx = ox - q0.x, ty = oy - q0.y, tz = oz - q0.z;
  const float u = (tx * px + ty * py + tz * pz) * invDet;
  if (u < 0.0f || u > 1.0f) return FSPT_MAX_T;
  const float qx = ty * e1z - e1y * tz, qy = tz * e1x - e1z * tx, qz = tx * e1y - e1x * ty;  // cross(t,e1)
  const float v = (dx * qx + dy * qy + dz * qz) * invDet;
  if (v < 0.0f || u + v > 1.0f) return FSPT_MAX_T;
  const float dist = (e2x * qx + e2y * qy + e2z * qz) * invDet;
  return dist > FSPT_EPSILON ? dist : FSPT_MAX_T;
}

// CAMERA = the primary launch of a render wave: the ray of slot `my` is generated on the fly (camera.fs) and the whole
// ray + hit record is written at retirement, so the camera pass, its 32 B/path of writes and this launch's
// record reads disappear.
// NODE_TEX = false: the node array is too large for a linear texture (2^27 texels), everything goes through the LSU.
// LIST (CAMERA only, adaptive sampling): path j * S + s renders the pixel of slot A.list[j].
template <bool WRITE_COUNT, bool CAMERA, bool NODE_TEX, bool LIST = false>
__global__ void __launch_bounds__(TRACE_THREADS, TRACE_MIN_BLOCKS) k_trace(const TraceArgs A) {
  const unsigned lane = threadIdx.x & 31u;
  const unsigned FULL = 0xffffffffu;
  // queue sizes: read once per CTA into shared memory.  (Re-reading them from global memory at every refill was a
  // measured 26 % regression: they share a sector with nothing hot any more, but any per-refill global load sits on
  // the critical path of the fetch.)
  __shared__ int s_counts[2];
  if (threadIdx.x == 0) { s_counts[0] = A.counts[0]; s_counts[1] = A.counts[1]; }
  __syncthreads();

  // Per-lane on-chip state, ONE shared array laid out [row][thread] (bank = lane for any per-lane row: conflict-free):
  //   rows 0..6  ray values that only one phase reads -- d (leaf steps), 1/d (interior steps), record position
  //              (retirement) -- so they stay out of the register file; their loads overlap the node / triangle fetch
  //              of the same step;
  //   rows 7..   the first TRACE_SMEM_STACK entries of the traversal stack; deeper entries spill to local memory.
  // `lane_addr` is the 32-bit shared-window address of the thread's column, `sp` the BYTE offset of its next free stack
  // entry inside the column (row * 4 * TRACE_THREADS), so one register is the depth and (plus lane_addr) the address, and
  // "still in shared memory" is a comparison with a constant.  Every access is an explicit ld.shared / st.shared on
  // [lane_addr + offset]: when the arrays were indexed through C++ pointers ptxas rebuilt the shared-window base
  // (S2R SR_CgaCtaId + 3 instructions) in front of every push and pop, on the pop -> node-fetch dependency chain.  The
  // address is passed through an opaque `mov` once so that it lives in one register instead of being rematerialised.
  constexpr int RAY_ROWS = 7;
  constexpr unsigned ROW = 4u * TRACE_THREADS;
  __shared__ int s_lane[(RAY_ROWS + TRACE_SMEM_STACK) * TRACE_THREADS];
  unsigned lane_addr;
  asm volatile("mov.u32 %0, %1;" : "=r"(lane_addr) : "r"((unsigned)__cvta_generic_to_shared(s_lane) + 4u * threadIdx.x));
#define LANE_LD(dst, off) asm volatile("ld.shared.b32 %0, [%1];" : "=r"(dst) : "r"(lane_addr + (off)))
#define LANE_ST(off, v) asm volatile("st.shared.b32 [%0], %1;" ::"r"(lane_addr + (off)), "r"(v))
  int spill[FSPT_STACK - TRACE_SMEM_STACK];
  constexpr unsigned SP0 = ROW * RAY_ROWS, SMEM_END = ROW * (RAY_ROWS + TRACE_SMEM_STACK);
#define STACK_PUSH(v)                                                              \
  do {                                                                             \
    const int v_ = (v);                                                            \
    if (sp < SMEM_END) LANE_ST(sp, v_);                                            \
    else spill[(sp - SMEM_END) / ROW] = v_;                                        \
    sp += ROW;                                                                     \
  } while (0)
#define STACK_POP(dst)                                                             \
  do {                                                                             \
    sp -= ROW;                                                                     \
    if (sp < SMEM_END) LANE_LD(dst, sp);                                           \
    else dst = spill[(sp - SMEM_END) / ROW];                                       \
  } while (0)
  int cur = FSPT_SENTINEL;
  unsigned sp = SP0;
  int cnt_exact = 0;  // visits of the current ray (the bvh_test count of the WRITE_COUNT variant)
  bool kind = false, have = false;
  enum { R_DX = 0, R_DY = 1, R_DZ = 2, R_IX = 3, R_IY = 4, R_IZ = 5, R_SLOT = 6 };
#define RAY_GET(row) ([&] { int v_; LANE_LD(v_, (row) * ROW); return v_; }())
#define RAY_GETF(row) __int_as_float(RAY_GET(row))
#define RAY_SET(row, v) LANE_ST((row) * ROW, (int)(v))
#define RAY_SETF(row, v) LANE_ST((row) * ROW, __float_as_int(v))
  float ox = 0, oy = 0, oz = 0;
  float tbest = FSPT_MAX_T;
  int ibest = -1;
  // interior / leaf visits of all rays this thread traces in one launch, one increment per step (one ray alone can pass
  // 2^16: a flat fan or a sliver soup gives 10^5).  The sums are exact while visits per ray times rays per thread per
  // launch stays below 2^32.
  unsigned n_interior = 0, n_leaves = 0;
  bool drained = false;
  bool boolean_ray = false;  // only hit-or-miss is consumed (tracer.fs:502, :509 at the last bounce)

  // start the ray whose two words are o4 / d4 on this lane
  auto start_ray = [&](const float4 o4, const float4 d4, int slot) {
    ox = o4.x; oy = o4.y; oz = o4.z;
    const float dx = d4.x, dy = d4.y, dz = d4.z;
    RAY_SET(R_SLOT, slot);
    RAY_SETF(R_DX, dx); RAY_SETF(R_DY, dy); RAY_SETF(R_DZ, dz);
    const float ix = 1.0f / dx, iy = 1.0f / dy, iz = 1.0f / dz;  // `vec3 inverse = 1.0 / ray.dir`, tracer.fs:318
    RAY_SETF(R_IX, ix); RAY_SETF(R_IY, iy); RAY_SETF(R_IZ, iz);
    have = true;
    tbest = FSPT_MAX_T; ibest = -1; cnt_exact = 0;
    sp = SP0;
    STACK_PUSH(FSPT_SENTINEL);
    cur = A.root_ref;
  };

  for (;;) {
    const bool need = (cur == FSPT_SENTINEL);
    const bool retire = need && have;
    if (retire) {  // retire the finished ray
      const int slot = RAY_GET(R_SLOT);
      if (CAMERA) {
        A.ps.ro(slot) = make_float4(ox, oy, oz, tbest);
        A.ps.rd(slot) = make_float4(RAY_GETF(R_DX), RAY_GETF(R_DY), RAY_GETF(R_DZ), __int_as_float(ibest));
      } else if (!kind) {
        A.ps.ro(slot).w = tbest;
        A.ps.rd(slot).w = __int_as_float(ibest);
      } else {
        A.ps.sh[slot] = (ibest == -1) ? 2 : 3;  // the record's shadow-state byte
      }
      if (WRITE_COUNT) A.count_out[slot] = cnt_exact;
      if (A.hit_flag && !kind) A.hit_flag[slot] = (ibest != -1);  // continuation rays: slot = queue position
      have = false;
    }
    if (!drained) {
      const unsigned m = __ballot_sync(FULL, need);
      if (m) {
        const int n_cont = s_counts[0], total = n_cont + s_counts[1];  // shared memory: two fewer live registers
        const int want = __popc(m);
        const int rank = __popc(m & ((1u << lane) - 1u));
        const int leader = __ffs(m) - 1;
        int base = 0;
        if ((int)lane == leader) base = atomicAdd(A.next, want);
        base = __shfl_sync(FULL, base, leader);
        if (base + want >= total) drained = true;
        const int my = base + rank;
        if (need && my < total) {
          if (CAMERA) {
            kind = false;
            v3 o, d;
            int px, py;
            camera_ray<LIST>(A.f, A.rb_cam, A.div_s, my, o, d, px, py, A.list);
            start_ray(make_float4(o.x, o.y, o.z, 0.0f), make_float4(d.x, d.y, d.z, 0.0f), my);
          } else {
            // continuation rays: words 0 / 1 of record `my`; shadow rays: their own dense array written by k_shade
            // (origin | record position, direction | -), no indirection through a list
            kind = my >= n_cont;
            const float4* src = kind ? A.shadow_rays + 2 * (size_t)(my - n_cont) : &A.ps.ro(my);
            const float4 o4 = src[0], d4 = src[1];
            // shadow rays always; continuation rays when k_shade marked the path's last bounce (index word = -2)
            boolean_ray = A.anyhit && (kind || __float_as_int(d4.w) == -2);
            start_ray(o4, d4, kind ? __float_as_int(o4.w) : my);
          }
        }
      }
    }
    if (__ballot_sync(FULL, cur != FSPT_SENTINEL) == 0u) break;

    const int refill = drained ? 1 : TRACE_REFILL;
    for (;;) {
      // Warp-level phase scheduling: every iteration runs ONE step for the larger group of lanes -- those
      // standing on an interior node or those standing on a leaf -- and the other group waits.  (A classic
      // while-while loop lets a few long interior walks hold the whole warp: measured 6.8 of 32 lanes active.)
      const bool is_int = cur >= 0;
      const bool is_leaf = !is_int && cur != FSPT_SENTINEL;
      const int ni = __popc(__ballot_sync(FULL, is_int)), nl = __popc(__ballot_sync(FULL, is_leaf));
      if (ni + nl < refill) break;
      if (ni >= nl) {
        // ---- interior node: both child boxes from one 64-byte record --------------------------------
        if (is_int) {
          if (WRITE_COUNT) cnt_exact++;
          n_interior++;
          // The record's four words are split between the two L1 data pipes (texture fetch / LSU load): the
          // kernel is bound by L1 wavefronts (ncu: l1tex data-pipe ~60 % busy), not by issue slots.  Measured with
          // 36 warps/SM: words 0,1 via TLD + words 2,3 via LDG is 0.5 % / 2.5 % faster than all four via TLD on the
          // 82 k / 1 M-triangle scenes; all four via LDG is 2 % / 11 % slower.
          const float4* np = A.nodes + 4 * (size_t)cur;
          const float4 a = NODE_TEX ? tex1Dfetch<float4>(A.nodes_tex, 4 * cur) : __ldg(np);
          const float4 b = NODE_TEX ? tex1Dfetch<float4>(A.nodes_tex, 4 * cur + 1) : __ldg(np + 1);
          const float4 c = __ldg(np + 2);
          const float4 df = __ldg(np + 3);
          const int cl = __float_as_int(df.x), cr = __float_as_int(df.y);
          float lh, rh;
          slab_pair(a, b, c, bc2(ox), bc2(oy), bc2(oz), bc2(RAY_GETF(R_IX)), bc2(RAY_GETF(R_IY)), bc2(RAY_GETF(R_IZ)), lh, rh);
          const bool tl = lh < tbest, tr = rh < tbest;
          const bool right_first = lh > rh;                   // tracer.fs:384 (ties go left)
          if (tl && tr) {
            STACK_PUSH(right_first ? cl : cr);                // deferred child, tracer.fs:391
            cur = right_first ? cr : cl;
          } else if (tl || tr) {
            cur = tl ? cl : cr;
          } else {
            STACK_POP(cur);
          }
        }
      } else {
        // ---- leaf: 4 consecutive triangles ----------------------------------------------------------
        if (is_leaf) {
          if (WRITE_COUNT) cnt_exact++;
          n_leaves++;
          const float dx = RAY_GETF(R_DX), dy = RAY_GETF(R_DY), dz = RAY_GETF(R_DZ);
          const int first = ~cur;
          const float4* tp = A.tris + 3 * (size_t)first;
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            // (through the LSU: with the triangle words on the texture pipe the traversal measured 2-4 % slower)
            const float4 q0 = __ldg(tp + 3 * k), q1 = __ldg(tp + 3 * k + 1), q2 = __ldg(tp + 3 * k + 2);
            const float res = tri_test(q0, q1, q2, ox, oy, oz, dx, dy, dz);
            if (res < tbest) { ibest = first + k; tbest = res; }
          }
          STACK_POP(cur);
          if (!CAMERA && boolean_ray && ibest != -1) cur = FSPT_SENTINEL;  // any hit settles it
        }
      }
    }
  }
  // per-warp statistics -> 3 atomics per warp
  unsigned long long s_nodes = (unsigned long long)n_interior + n_leaves, s_leaves = n_leaves;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    s_nodes += __shfl_xor_sync(FULL, s_nodes, o);
    s_leaves += __shfl_xor_sync(FULL, s_leaves, o);
  }
  if (lane == 0) {
    atomicAdd(A.stats + 1, s_nodes);
    atomicAdd(A.stats + 2, s_leaves);
  }
  // every queue item is one ray and every item is traced exactly once
  if (blockIdx.x == 0 && threadIdx.x == 0) atomicAdd(A.stats + 0, (unsigned long long)(A.counts[0] + A.counts[1]));
#undef STACK_PUSH
#undef STACK_POP
#undef LANE_LD
#undef LANE_ST
#undef RAY_GET
#undef RAY_GETF
#undef RAY_SET
#undef RAY_SETF
}
