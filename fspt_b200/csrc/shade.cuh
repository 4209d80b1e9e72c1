// shade.cuh -- camera ray generation, per-vertex shading (UE4-style GGX / Lambert / refraction + Beer,
// env-map NEE with MIS) and accumulation, as wavefront stages around the traversal kernel.
//
// Replaces camera.fs main (:37-46) and tracer.fs main (:436-518) minus its three intersectScene calls.
// The reference runs a whole path inside one fragment invocation; here a path is a slot of PathState that
// alternates between k_shade (one vertex) and k_trace (its shadow + continuation rays).  Per path the
// floating-point operations and their order are the reference's, so per-sample colours are bit-identical
// to the CPU oracle (DESIGN.md section 4); only the scheduling differs.
#pragma once
#include "device_common.cuh"
#include "dm_math.cuh"

#include "camera.cuh"

// ---------------------------------------------------------------------------------------------------------
// camera.fs main as a stand-alone pass (mode=test / fspt_debug_primary; the render loop fuses ray generation into
// the primary traversal launch, see traverse.cuh).  One thread per path slot.
__global__ void __launch_bounds__(256) k_camera(const FrameParams f, const float* __restrict__ rb_cam, int n_paths,
                                                FastDiv div_s, PathState ps, float4* cam_pos_out,
                                                float4* cam_dir_out) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= n_paths) return;
  v3 o, d;
  int x, y;
  camera_ray(f, rb_cam, div_s, p, o, d, x, y);
  ps.ro(p) = make_float4(o.x, o.y, o.z, FSPT_MAX_T);
  ps.rd(p) = make_float4(d.x, d.y, d.z, __int_as_float(-1));
  if (cam_pos_out) {  // frame-sized targets
    const size_t px = (size_t)(y + f.ry0) * f.width + (size_t)(x + f.rx0);
    cam_pos_out[px] = make_float4(o.x, o.y, o.z, 1.0f);
    cam_dir_out[px] = make_float4(d.x, d.y, d.z, 1.0f);
  }
}

// ---------------------------------------------------------------------------------------------------------
// Texture units.  The atlas and the environment are CUDA texture objects (block-linear arrays through the
// texture cache); texels are fetched un-filtered and the GL LINEAR weights (GL ES 3.0 section 3.8.10) are
// applied in f32 exactly as the oracle does, because hardware filtering uses 8-bit fixed-point weights.
// unorm8 -> f32 is (float)c / 255.0f; the 256 possible quotients are computed once per block with IEEE division
// into shared memory, so a bilinear fetch costs 16 LDS instead of 16 I2F + 16 division sequences (XU pipe).
extern __shared__ float s_unorm8[];
__device__ __forceinline__ void init_unorm8_lut() {
  for (int i = threadIdx.x; i < 256; i += blockDim.x) s_unorm8[i] = (float)i / 255.0f;
  __syncthreads();
}
__device__ __forceinline__ float4 texel8(uchar4 c) {
  return make_float4(s_unorm8[c.x], s_unorm8[c.y], s_unorm8[c.z], s_unorm8[c.w]);
}
__device__ __forceinline__ float4 bilerp(float4 t00, float4 t10, float4 t01, float4 t11, float a, float b) {
  const float w00 = (1.0f - a) * (1.0f - b), w10 = a * (1.0f - b), w01 = (1.0f - a) * b, w11 = a * b;
  float4 r;
  r.x = w00 * t00.x + w10 * t10.x + w01 * t01.x + w11 * t11.x;
  r.y = w00 * t00.y + w10 * t10.y + w01 * t01.y + w11 * t11.y;
  r.z = w00 * t00.z + w10 * t10.z + w01 * t01.z + w11 * t11.z;
  r.w = w00 * t00.w + w10 * t10.w + w01 * t01.w + w11 * t11.w;
  return r;
}
// texel index wrapping.  coord_to_int() bounds |i| by 1e9, so 32-bit arithmetic is exact; power-of-two sizes
// (every atlas / environment in practice) wrap with a mask, which equals the mathematical modulo for negatives too.
__device__ __forceinline__ int wrap_repeat(int i, int size) {
  if ((size & (size - 1)) == 0) return i & (size - 1);
  int m = i % size;
  if (m < 0) m += size;
  return m;
}
__device__ __forceinline__ int wrap_clamp(int i, int size) { return i < 0 ? 0 : (i >= size ? size - 1 : i); }

// The four texture(texArray, vec3(uv, layer)) lookups of one vertex (tracer.fs:453-456): REPEAT/REPEAT, LINEAR
// (main.js:551-555).  All four maps share the texel footprint, so the coordinates are computed once and the 16
// fetches are issued back to back (one memory round trip instead of four).
// Colour layers (TexturePacker.addColor, texture_packer.js:25-34,152-157) are res x res copies of one texel: their
// taps are known without touching the 16.8 MB layer; the filter arithmetic still runs, so the f32 result is the
// one the fetches would give.
__device__ __forceinline__ int atlas_layer(float layerf, int n_layers) {
  const long long Lq = coord_to_int(floorf(layerf + 0.5f));
  return (int)(Lq < 0 ? 0 : (Lq >= n_layers ? n_layers - 1 : Lq));
}
__device__ __forceinline__ uchar4 as_uchar4(unsigned v) { return make_uchar4(v & 0xff, (v >> 8) & 0xff, (v >> 16) & 0xff, v >> 24); }
__device__ __forceinline__ void texture_atlas4(const DeviceScene& sc, float u, float v, const float (&layerf)[4], float4 (&out)[4]) {
  const int R = sc.atlas_res;
  const float x = u * (float)R - 0.5f, y = v * (float)R - 0.5f;
  const float fx = floorf(x), fy = floorf(y);
  const float a = x - fx, b = y - fy;
  const int ixx = coord_to_i32(fx), iyy = coord_to_i32(fy);
  const float i0 = (float)wrap_repeat(ixx, R) + 0.5f, i1 = (float)wrap_repeat(ixx + 1, R) + 0.5f;
  const float j0 = (float)wrap_repeat(iyy, R) + 0.5f, j1 = (float)wrap_repeat(iyy + 1, R) + 0.5f;
  int L[4];
  uint2 info[4];
#pragma unroll
  for (int m = 0; m < 4; ++m) {
    L[m] = atlas_layer(layerf[m], sc.atlas_layers);
    info[m] = __ldg(sc.layer_info + L[m]);
  }
  uchar4 t[4][4];
#pragma unroll
  for (int m = 0; m < 4; ++m) {
    t[m][0] = t[m][1] = t[m][2] = t[m][3] = as_uchar4(info[m].y);
    if (!info[m].x) {
      t[m][0] = tex2DLayered<uchar4>(sc.atlas, i0, j0, L[m]);
      t[m][1] = tex2DLayered<uchar4>(sc.atlas, i1, j0, L[m]);
      t[m][2] = tex2DLayered<uchar4>(sc.atlas, i0, j1, L[m]);
      t[m][3] = tex2DLayered<uchar4>(sc.atlas, i1, j1, L[m]);
    }
  }
#pragma unroll
  for (int m = 0; m < 4; ++m) out[m] = bilerp(texel8(t[m][0]), texel8(t[m][1]), texel8(t[m][2]), texel8(t[m][3]), a, b);
}
// Same four lookups from the material-interleaved atlas (device_common.cuh "MatTexel"): one 16-byte fetch per tap
// carries the texel of all four maps.  All-constant materials (four colour layers) need no fetch at all.
__device__ __forceinline__ void texture_material(const DeviceScene& sc, float u, float v, int mat, float4 (&out)[4]) {
  const int R = sc.atlas_res;
  const float x = u * (float)R - 0.5f, y = v * (float)R - 0.5f;
  const float fx = floorf(x), fy = floorf(y);
  const float a = x - fx, b = y - fy;
  const int4 info = __ldg(sc.mat_info + 2 * mat);
  uint4 t00, t10, t01, t11;
  if (info.x >= 0) {
    const int ixx = coord_to_i32(fx), iyy = coord_to_i32(fy);
    const float i0 = (float)wrap_repeat(ixx, R) + 0.5f, i1 = (float)wrap_repeat(ixx + 1, R) + 0.5f;
    const float j0 = (float)wrap_repeat(iyy, R) + 0.5f, j1 = (float)wrap_repeat(iyy + 1, R) + 0.5f;
    t00 = tex2DLayered<uint4>(sc.mat_tex, i0, j0, info.x);
    t10 = tex2DLayered<uint4>(sc.mat_tex, i1, j0, info.x);
    t01 = tex2DLayered<uint4>(sc.mat_tex, i0, j1, info.x);
    t11 = tex2DLayered<uint4>(sc.mat_tex, i1, j1, info.x);
  } else {
    const int4 info2 = __ldg(sc.mat_info + 2 * mat + 1);
    t00 = make_uint4((unsigned)info.y, (unsigned)info.z, (unsigned)info.w, (unsigned)info2.x);
    t10 = t01 = t11 = t00;
  }
  out[0] = bilerp(texel8(as_uchar4(t00.x)), texel8(as_uchar4(t10.x)), texel8(as_uchar4(t01.x)), texel8(as_uchar4(t11.x)), a, b);
  out[1] = bilerp(texel8(as_uchar4(t00.y)), texel8(as_uchar4(t10.y)), texel8(as_uchar4(t01.y)), texel8(as_uchar4(t11.y)), a, b);
  out[2] = bilerp(texel8(as_uchar4(t00.z)), texel8(as_uchar4(t10.z)), texel8(as_uchar4(t01.z)), texel8(as_uchar4(t11.z)), a, b);
  out[3] = bilerp(texel8(as_uchar4(t00.w)), texel8(as_uchar4(t10.w)), texel8(as_uchar4(t01.w)), texel8(as_uchar4(t11.w)), a, b);
}
// texture(envTex, c): S REPEAT, T CLAMP_TO_EDGE, LINEAR on the ENCODED RGBE texel (main.js:170-180)
__device__ __forceinline__ float4 texture_env(cudaTextureObject_t env, int W, int H, float u, float v) {
  const float x = u * (float)W - 0.5f, y = v * (float)H - 0.5f;
  const float fx = floorf(x), fy = floorf(y);
  const float a = x - fx, b = y - fy;
  const int ixx = coord_to_i32(fx), iyy = coord_to_i32(fy);
  const float i0 = (float)wrap_repeat(ixx, W) + 0.5f, i1 = (float)wrap_repeat(ixx + 1, W) + 0.5f;
  const float j0 = (float)wrap_clamp(iyy, H) + 0.5f, j1 = (float)wrap_clamp(iyy + 1, H) + 0.5f;
  const uchar4 t00 = tex2D<uchar4>(env, i0, j0), t10 = tex2D<uchar4>(env, i1, j0);
  const uchar4 t01 = tex2D<uchar4>(env, i0, j1), t11 = tex2D<uchar4>(env, i1, j1);
  return bilerp(texel8(t00), texel8(t10), texel8(t01), texel8(t11), a, b);
}
// envColor + envSample, tracer.fs:410-419
__device__ __noinline__ v3 env_sample_(cudaTextureObject_t env, int W, int H, float dx, float dy, float dz, float envTheta) {
  const float cx = envTheta + dm::atan2f_(dz, dx) / FSPT_TAU;
  const float cy = dm::asinf_(-dy) * FSPT_INV_PI + 0.5f;
  const float4 rgbe = texture_env(env, W, H, cx, cy);
  // pow(2.0, e), tracer.fs:412: in FSPT-DM2 log2(2.0) evaluates to exactly 1.0, so this is exp2(e) bit for bit
  const float p = dm::exp2f_(rgbe.w * 255.0f - 128.0f);
  return mk3(rgbe.x * p, rgbe.y * p, rgbe.z * p);
}
__device__ __forceinline__ v3 env_sample(const DeviceScene& sc, v3 dir, float envTheta) {
  return env_sample_(sc.env, sc.env_w, sc.env_h, dir.x, dir.y, dir.z, envTheta);
}

// ---- BSDF pieces, tracer.fs:194-298 ---------------------------------------------------------------------
__device__ __forceinline__ v2 mis_weights(float a, float b) {
  v2 r;
  if (a > FSPT_EPSILON && b > FSPT_EPSILON) {
    const float a2 = a * a, b2 = b * b, a2b2 = a2 + b2;
    r.x = a2 / a2b2;
    r.y = b2 / a2b2;
  } else {
    r.x = 1.0f;
    r.y = 0.0f;
  }
  return r;
}
__device__ __forceinline__ float gtr2(float ndh, float a) {
  const float a2 = a * a;
  const float t = 1.0f + (a2 - 1.0f) * ndh * ndh;
  return a2 / (FSPT_PI * t * t);
}
__device__ __forceinline__ float smith_g(float NDotv, float alphaG) {
  const float a = alphaG * alphaG;
  const float b = NDotv * NDotv;
  return 1.0f / (NDotv + sqrtf(a + b - a * b));
}
__device__ __forceinline__ float gtr2_pdf(v3 incident, v3 normal, v2 mr, v3 bsdfDir) {
  const float specularAlpha = fmaxf(0.001f, mr.y);
  const v3 halfVec = normalize(add(bsdfDir, incident));
  const float cosTheta = fabsf(dot(halfVec, normal));
  const float pdfgtr2 = gtr2(cosTheta, specularAlpha) * cosTheta;
  return pdfgtr2 / (4.0f * fabsf(dot(bsdfDir, halfVec)));
}
__device__ __forceinline__ float schlick(v3 incident, v3 normal, v2 ns) {
  float r0 = div_z(ns.x - ns.y, ns.x + ns.y);  // ior 1 gives 0 / 2
  r0 *= r0;
  float cosTheta = dot(normal, incident);
  if (ns.x > ns.y) {
    const float n = ns.x / ns.y;
    const float sinTheta2 = n * n * (1.0f - cosTheta * cosTheta);
    if (sinTheta2 > 1.0f) return 1.0f;
    cosTheta = sqrtf(1.0f - sinTheta2);
  }
  const float x = 1.0f - cosTheta;
  return r0 + (1.0f - r0) * x * x * x * x * x;
}
__device__ __forceinline__ v3 eval_specular(v3 incident, v3 normal, v3 diffuseColor, v2 mr, v3 bsdfDir) {
  const float ndl = dot(normal, bsdfDir);
  const float ndv = dot(normal, incident);
  const v3 H = normalize(add(bsdfDir, incident));
  const float ndh = dot(normal, H);
  const float a = fmaxf(0.001f, mr.y);
  const float Ds = gtr2(ndh, a);
  const v3 Fs = mix3(mk3(1.0f, 1.0f, 1.0f), diffuseColor, mr.x);
  float roughg = (mr.y * 0.5f + 0.5f);
  roughg = roughg * roughg;
  const float Gs = smith_g(ndl, roughg) * smith_g(ndv, roughg);
  return mul(mul(Gs, Fs), Ds);
}
__device__ __forceinline__ void tangent_frame(v3 normal, v3& tangent, v3& bitangent) {  // tracer.fs:259-261
  const v3 up = fabsf(normal.z) < 0.999f ? mk3(0.0f, 0.0f, 1.0f) : mk3(1.0f, 0.0f, 0.0f);
  const v3 t = cross(up, normal);  // one component is exactly 0 (up is an axis): keep it out of the divide sequence
  tangent = div_z(t, length(t));
  bitangent = cross(normal, tangent);
}

struct ShadeArgs {
  DeviceScene sc;
  PathState ps;               // records of the paths to shade, dense: position 0 .. counts_in[0]-1
  PathState ps_out;           // compacted records of the paths that continue (position = append order)
  FrameParams f;
  const float* rb_trace;      // per sample-in-wave
  const int* counts_in;       // [0] = number of records in ps
  float4* shadow_rays_out;    // shadow rays of the paths that cast one, dense, 2 words each: origin | position in ps_out,
                              // direction | -.  (A list of record positions made the traversal kernel's shadow-ray
                              // fetch two dependent gathers over two sectors; this is one contiguous 32-byte read.)
  int* counts_out;            // [0] continuation, [1] shadow
  int* tile_next;             // tile cursor, 0 between launches (k_shade resets it); on a 128-byte line of its own
  float4* sample_color;       // [pixel][sample-in-wave] final un-clamped path colour
  unsigned long long* capped; // paths stopped by the refraction cap
  int n_samples;              // samples in flight in this wave (slot = pixel * n_samples + sample)
  FastDiv div_s;              // by n_samples
  int first;                  // 1: slots hold fresh primary rays (tracer.fs:440-445)
  int max_refractions;
  int anyhit;
  const unsigned char* hit_flag;  // hit / miss per record position, written by k_trace.  (Measured and dropped: a 4-byte hit
                                  // INDEX per position carried through the queues, so that the shading records are requested
                                  // together with the path record -- shade +2.4 %: wider reads and queues cost more than
                                  // the shorter dependent chain saves at 32 warps/SM.  Also measured and dropped: requesting
                                  // the NEXT tile's bytes before this tile's groups are shaded, +0.5 %.)
  const int* list;            // LIST: the slots of the pixels this wave renders (adaptive.cuh); last, so that the other
                              // instantiations keep their parameter offsets and instructions
};

// Warp-aggregated append: one atomicAdd per warp per list (ballot + popc prefix); call with all 32 lanes
__device__ __forceinline__ void append(bool want, int value, int* list, int* counter) {
  const unsigned m = __ballot_sync(0xffffffffu, want);
  if (!want) return;
  const unsigned lane = threadIdx.x & 31u;
  const int leader = __ffs(m) - 1;
  int base = 0;
  if ((int)lane == leader) base = atomicAdd(counter, __popc(m));
  base = __shfl_sync(m, base, leader);
  list[base + __popc(m & ((1u << lane) - 1u))] = value;
}

// position of this lane's element when the lanes with `want` append to a dense array (one atomicAdd per warp)
__device__ __forceinline__ int append_pos(bool want, int* counter) {
  const unsigned m = __ballot_sync(0xffffffffu, want);
  if (m == 0u) return 0;
  const unsigned lane = threadIdx.x & 31u;
  const int leader = __ffs(m) - 1;
  int base = 0;
  if ((int)lane == leader) base = atomicAdd(counter, __popc(m));
  base = __shfl_sync(0xffffffffu, base, leader);
  return base + __popc(m & ((1u << lane) - 1u));
}

template <bool LIST>
__device__ __forceinline__ void write_sample(const ShadeArgs& A, int slot, v3 color) {
  const int j = (int)fast_div((unsigned)slot, A.div_s), s = slot - j * A.n_samples;
  int x, y;
  path_to_pixel(A.f, LIST ? A.list[j] : j, x, y);
  // [pixel][sample]: the samples of a pixel finish in adjacent lanes and land in adjacent 16-byte entries
  A.sample_color[((size_t)y * A.f.rw + x) * A.n_samples + s] = make_float4(color.x, color.y, color.z, 1.0f);
}

// The tail of the previous loop iteration for a path whose ray MISSED: tracer.fs:442-443 (primary) or
// :502-504 + :508-512 (bounce).  Ends the path.
template <bool LIST>
__device__ __forceinline__ void shade_miss(const ShadeArgs& A, int pos) {
  const int slot_in = pos;  // record position in A.ps
  int slot = pos;           // path identity (pixel * S + sample); equals the position only in the first pass
  const float4 d4 = A.ps.rd(slot_in);
  const v3 rayDir = mk3(d4.x, d4.y, d4.z);
  const v3 env = env_sample(A.sc, rayDir, A.f.env_theta);
  v3 color;
  if (A.first) {
    color = add(mk3(0.0f, 0.0f, 0.0f), env);  // :443
  } else {
    const float4 c4 = A.ps.col(slot_in), t4 = A.ps.thr(slot_in);
    slot = __float_as_int(c4.w);
    color = mk3(c4.x, c4.y, c4.z);
    if (A.ps.sh[slot_in] == 2) {  // shadow.index == -1, :502-504
      const float4 p4 = A.ps.pend(slot_in);
      color = add(color, mk3(p4.x, p4.y, p4.z));
    }
    const v3 reflectance = mk3(t4.x, t4.y, t4.z);                 // accumulatedReflectance *= bsdfThroughput (:508) was
    color = add(color, mul(mul(reflectance, env), t4.w));         // folded into the stored value; :510
  }
  write_sample<LIST>(A, slot, color);
}

// One loop iteration of tracer.fs main (:446-513) for a path whose ray HIT, split at the intersectScene calls.
// Returns true when the path continues; `out` then holds its new record (words 0, 1, 3, 4, 5 = the five words of the
// record in HBM) and, in word 2, the shadow ray's direction for the dense shadow-ray array.
struct PathRecord { float4 w[6]; };
__device__ __forceinline__ void store_record(const PathState& ps, int pos, const PathRecord& rec, bool shadow) {
  float4* dst = ps.rec + FSPT_PATH_WORDS * (size_t)pos;
  dst[0] = rec.w[0]; dst[1] = rec.w[1]; dst[2] = rec.w[3]; dst[3] = rec.w[4]; dst[4] = rec.w[5];
  ps.sh[pos] = shadow ? 1 : 0;  // (every record: a stale 2 of an earlier bounce must not survive at this position)
}
template <bool MAT_TEX, bool LIST>
__device__ __forceinline__ bool shade_hit(const ShadeArgs& A, int pos, bool& shadow, PathRecord& out) {
  const DeviceScene& sc = A.sc;
  int slot = pos;  // path identity; equals the record position only in the first pass
  const float4 o4 = A.ps.ro(pos), d4 = A.ps.rd(pos);
  v3 rayOrigin = mk3(o4.x, o4.y, o4.z), rayDir = mk3(d4.x, d4.y, d4.z);
  const float hit_t = o4.w;
  const int hit_index = __float_as_int(d4.w);
  const float envTheta = A.f.env_theta;
  v3 color, reflectance;
  int i = 0, refractions = 0;
  shadow = false;
  if (A.first) {
    color = mk3(0.0f, 0.0f, 0.0f);
    reflectance = mk3(1.0f, 1.0f, 1.0f);
  } else {
    const float4 c4 = A.ps.col(pos), t4 = A.ps.thr(pos);
    const float4 p4 = A.ps.pend(pos);
    const int shadow_state = A.ps.sh[pos];
    slot = __float_as_int(c4.w);
    color = mk3(c4.x, c4.y, c4.z);
    reflectance = mk3(t4.x, t4.y, t4.z);  // already multiplied by the previous bsdfThroughput (:508), see the store below
    const int packed = __float_as_int(p4.w);
    i = (packed & 0xffff) - 0x100;  // stored biased so that i = -1 survives
    refractions = packed >> 16;
    if (shadow_state == 2) color = add(color, mk3(p4.x, p4.y, p4.z));  // shadow.index == -1, :502-504
    ++i;                                                    // for (...; ++i), :446
    if (!(i < FSPT_NUM_BOUNCES)) {
      write_sample<LIST>(A, slot, color);
      return false;
    }
  }
  const float randBase = A.rb_trace[slot - (int)fast_div((unsigned)slot, A.div_s) * A.n_samples];
  // createMaterial / createTriangle / createTexCoords / createNormals, :447-449,460
  const float4* rec = sc.shade + 12 * (size_t)hit_index;
  const float4 m0 = __ldg(rec), m2 = __ldg(rec + 2);
  const float4 u0 = __ldg(rec + 3), u1 = __ldg(rec + 4);
  const float mapDiffuse = m0.x, mapSpecular = m0.y, mapNormal = m0.z, mapRoughness = m0.w;
  const float matIor = m2.y, matDielectric = m2.z;
  const float4* tp = sc.tris + 3 * (size_t)hit_index;
  const float4 q0 = __ldg(tp), q1 = __ldg(tp + 1), q2 = __ldg(tp + 2);
  const v3 tv1 = mk3(q0.x, q0.y, q0.z);
  const v3 origin = add(rayOrigin, mul(rayDir, hit_t));  // :450
  // barycentricWeights, :339-353 (v0 = v2 - v1 and v1 = v3 - v1 are the stored edges)
  const v3 e0 = mk3(q0.w, q1.x, q1.y), e1 = mk3(q1.z, q1.w, q2.x), e2 = sub(origin, tv1);
  const float d00 = dot(e0, e0), d01 = dot(e0, e1), d11 = dot(e1, e1), d20 = dot(e2, e0), d21 = dot(e2, e1);
  const float invDenom = 1.0f / (d00 * d11 - d01 * d01);
  const float bv = (d11 * d20 - d01 * d21) * invDenom;
  const float bw_ = (d00 * d21 - d01 * d20) * invDenom;
  const float bu = 1.0f - bv - bw_;
  const float tcx = bu * u0.x + bv * u0.z + bw_ * u1.x;  // barycentricTexCoord, :328-330
  const float tcy = bu * u0.y + bv * u0.w + bw_ * u1.y;
  const float layers[4] = {mapDiffuse, mapSpecular, mapRoughness, mapNormal};
  float4 tex[4];
  if (MAT_TEX) texture_material(sc, tcx, tcy, __float_as_int(u1.z), tex);  // :453-456
  else texture_atlas4(sc, tcx, tcy, layers, tex);
  const float4 tD = tex[0], tE = tex[1], tMR = tex[2], tN = tex[3];
  const v3 texDiffuse = mk3(tD.x, tD.y, tD.z), texEmmissive = mk3(tE.x, tE.y, tE.z);
  v2 texMR;
  texMR.x = tMR.x;
  texMR.y = tMR.y;
  const v3 texNormal = mul(sub(mk3(tN.x, tN.y, tN.z), mk3(0.5f, 0.5f, 0.0f)), mk3(2.0f, 2.0f, 1.0f));
  texMR.y *= texMR.y;  // :457
  float seed = origin.x * randBase * origin.y * 1.396529836f + origin.z * 4761.52835f;  // :458
  // normals record: [n1 t1 b1 n2 t2 b2 n3 t3 b3] = floats 20..46 of the 48-float record
  float nn[28];
#pragma unroll
  for (int k = 0; k < 7; ++k) {
    const float4 t = __ldg(rec + 5 + k);
    nn[4 * k + 0] = t.x; nn[4 * k + 1] = t.y; nn[4 * k + 2] = t.z; nn[4 * k + 3] = t.w;
  }
  const v3 n1 = mk3(nn[0], nn[1], nn[2]), t1 = mk3(nn[3], nn[4], nn[5]), b1 = mk3(nn[6], nn[7], nn[8]);
  const v3 n2 = mk3(nn[9], nn[10], nn[11]), t2 = mk3(nn[12], nn[13], nn[14]), b2 = mk3(nn[15], nn[16], nn[17]);
  const v3 n3 = mk3(nn[18], nn[19], nn[20]), t3 = mk3(nn[21], nn[22], nn[23]), b3 = mk3(nn[24], nn[25], nn[26]);
  const v3 baryNormal = add(add(mul(bu, n1), mul(bv, n2)), mul(bw_, n3));  // :333-336
  const v3 baryTangent = add(add(mul(bu, t1), mul(bv, t2)), mul(bw_, t3));
  const v3 baryBiTangent = add(add(mul(bu, b1), mul(bv, b2)), mul(bw_, b3));
  v3 macroNormal = normalize(add(add(mul(texNormal.x, baryTangent), mul(texNormal.y, baryBiTangent)),
                                 mul(texNormal.z, baryNormal)));
  const bool inside = dot(neg(rayDir), baryNormal) < 0.0f;  // :461
  v2 ns;
  if (inside) { ns.x = matIor; ns.y = 1.0f; } else { ns.x = 1.0f; ns.y = matIor; }  // :462
  macroNormal = inside ? neg(macroNormal) : macroNormal;                          // :463
  rayOrigin = add(origin, mul(mul(macroNormal, FSPT_EPSILON), 2.0f));              // :464
  color = add(color, mul(mul(mul(reflectance, texEmmissive), texDiffuse), 30.0f));  // :467
  const v3 incident = neg(rayDir);
  v3 envThroughput, bsdfThroughput;
  float bsdfPdf;
  // sampleMicrofacet, :256-270
  v3 microNormal;
  {
    const float r1 = rnd(seed), r2 = rnd(seed);
    v3 tangent, bitangent;
    tangent_frame(macroNormal, tangent, bitangent);
    const float a = fmaxf(0.001f, texMR.y);
    const float phi = r1 * FSPT_TAU;
    const float cosTheta = sqrtf((1.0f - r2) / (1.0f + (a * a - 1.0f) * r2));
    const float sinTheta = clampf(sqrtf(1.0f - (cosTheta * cosTheta)), 0.0f, 1.0f);
    float sinPhi, cosPhi;
    dm::sincosf_(phi, sinPhi, cosPhi);
    const v3 h = mk3(sinTheta * cosPhi, sinTheta * sinPhi, cosTheta);
    microNormal = add(add(mul(tangent, h.x), mul(bitangent, h.y)), mul(macroNormal, h.z));
  }
  // sampleEnv, :421-434
  v3 envDir;
  float envPdf;
  {
    int idx = coord_to_i32((float)sc.n_bins * rnd(seed));
    if (idx >= sc.n_bins) idx = sc.n_bins - 1;
    if (idx < 0) idx = 0;
    const float4 bin = __ldg(sc.bins + idx);
    const float dimsx = (float)sc.env_w, dimsy = (float)sc.env_h;
    const float r1 = rnd(seed);
    const float r2 = rnd(seed);
    const float qx = (bin.z - bin.x) * r1 + bin.x, qy = (bin.w - bin.y) * r2 + bin.y;
    // division by a power of two = multiplication by its exact reciprocal, bit for bit (no divide sequence)
    const float uvx = -envTheta + (sc.env_pow2 ? qx * sc.inv_env_w : qx / dimsx);
    const float uvy = 0.0f + (sc.env_pow2 ? qy * sc.inv_env_h : qy / dimsy);
    const float theta = uvx * FSPT_TAU;
    const float phi = uvy * FSPT_PI;
    float sinPhi, cosPhi, sinTheta, cosTheta;
    dm::sincosf_(phi, sinPhi, cosPhi);
    dm::sincosf_(theta, sinTheta, cosTheta);
    envDir = mk3(cosTheta * sinPhi, cosPhi, sinTheta * sinPhi);
    const float nominal = sc.env_nominal;  // (dimsx * dimsy) / float(n_bins), evaluated once on the host
    envPdf = nominal / ((bin.z - bin.x) * (bin.w - bin.y) * FSPT_TAU * FSPT_PI * sinPhi);
  }
  const float cosEnv = dot(macroNormal, envDir);  // :474
  const bool specular = mixf(schlick(incident, microNormal, ns), 1.0f, texMR.x) > rnd(seed);  // :475
  if (specular) {
    rayDir = reflect(neg(incident), microNormal);  // :477
    bsdfPdf = gtr2_pdf(incident, macroNormal, texMR, rayDir);
    bsdfThroughput = div_z(mul(eval_specular(incident, macroNormal, texDiffuse, texMR, rayDir),
                             clampf(dot(macroNormal, rayDir), 0.0f, 1.0f)), bsdfPdf);
    envThroughput = div_z(mul(eval_specular(incident, macroNormal, texDiffuse, texMR, envDir),
                            clampf(cosEnv, 0.0f, 1.0f)), envPdf);
  } else if (matDielectric >= 0.0f) {  // :481-488
    bsdfPdf = 1.0f;
    bsdfThroughput = mk3(1.0f, 1.0f, 1.0f);
    envThroughput = mk3(0.0f, 0.0f, 0.0f);
    rayOrigin = sub(origin, mul(mul(macroNormal, FSPT_EPSILON), 2.0f));
    rayDir = refract(neg(incident), microNormal, ns.x / ns.y);
    i--;
    if (++refractions > A.max_refractions) {  // safety cap of the reference's unbounded loop
      i = FSPT_NUM_BOUNCES;
      atomicAdd(A.capped, 1ull);
    }
  } else {  // :489-494
    {
      const float r1 = rnd(seed), r2 = rnd(seed);
      v3 tangent, bitangent;
      tangent_frame(macroNormal, tangent, bitangent);
      const float r = sqrtf(r1);
      const float phi = FSPT_TAU * r2;
      float sp_, cp_;
      dm::sincosf_(phi, sp_, cp_);
      v3 dir;
      dir.x = r * cp_;
      dir.y = r * sp_;
      dir.z = sqrtf(fmaxf(0.0f, 1.0f - dir.x * dir.x - dir.y * dir.y));
      rayDir = add(add(mul(tangent, dir.x), mul(bitangent, dir.y)), mul(macroNormal, dir.z));
    }
    bsdfPdf = fabsf(dot(rayDir, macroNormal)) * FSPT_INV_PI;  // lambertPdf, :235-237
    const v3 lam = mul(texDiffuse, FSPT_INV_PI);               // evalLambert, :296-298
    bsdfThroughput = div_z(mul(lam, clampf(dot(macroNormal, rayDir), 0.0f, 1.0f)), bsdfPdf);
    envThroughput = div_z(mul(lam, clampf(cosEnv, 0.0f, 1.0f)), envPdf);
  }
  if (inside) {  // Beer's-law override, :497
    const v3 om_ = sub(mk3(1.0f, 1.0f, 1.0f), texDiffuse);
    const v3 b = sub(mk3(1.0f, 1.0f, 1.0f), mul(mul(om_, hit_t), matDielectric));
    bsdfThroughput = mk3(fmaxf(b.x, 0.0f), fmaxf(b.y, 0.0f), fmaxf(b.z, 0.0f));
  }
  const v2 weights = mis_weights(envPdf, bsdfPdf);  // :499
  shadow = (matDielectric < 0.0f && cosEnv > 0.0f);  // :500
  v3 pend = mk3(0.0f, 0.0f, 0.0f);
  if (shadow) pend = mul(mul(mul(reflectance, envThroughput), env_sample(sc, envDir, envTheta)), weights.x);  // :503
  out.w[0] = make_float4(rayOrigin.x, rayOrigin.y, rayOrigin.z, FSPT_MAX_T);
  // last bounce: the loop ends after this continuation ray whatever it hits (:446 with ++i), only hit-or-miss
  // matters (:509), so the traversal may stop at the first intersection (index word -2 = "boolean ray")
  const bool last_bounce = A.anyhit && (i + 1 >= FSPT_NUM_BOUNCES);
  out.w[1] = make_float4(rayDir.x, rayDir.y, rayDir.z, __int_as_float(last_bounce ? -2 : -1));
  out.w[2] = make_float4(envDir.x, envDir.y, envDir.z, __int_as_float(shadow ? 1 : 0));
  // accumulatedReflectance *= bsdfThroughput (:508) is a pure product of two values known here: storing it now gives
  // the same f32 bits as multiplying in the next pass and keeps the record small (five words in HBM)
  const v3 next_reflectance = mul(reflectance, bsdfThroughput);
  out.w[3] = make_float4(next_reflectance.x, next_reflectance.y, next_reflectance.z, weights.y);
  out.w[4] = make_float4(pend.x, pend.y, pend.z, __int_as_float(((i + 0x100) & 0xffff) | (refractions << 16)));
  out.w[5] = make_float4(color.x, color.y, color.z, __int_as_float(slot));  // the path's identity travels with it
  return true;
}

#ifndef SHADE_THREADS
#define SHADE_THREADS 256
#endif
#ifndef SHADE_MIN_BLOCKS
#define SHADE_MIN_BLOCKS 4  // 64 registers, 32 warps/SM.  Measured shading time vs 128 threads x 6 blocks (80 regs):
                            // 128x5 +8 %, 128x7 -7 %, 128x8 -5.5 %, 224x4 -8 %, 256x4 -9 %, 448x2 -3 %, 64x14 -5.5 %
#endif
// Path state is STREAM-COMPACTED every bounce: this kernel reads the dense record array the traversal just worked on
// (position i = i-th surviving path, in roughly ascending pixel order) and writes the records of the paths that
// continue to the next free positions of a second array, so record traffic is sequential in both kernels and no
// index lists exist except for shadow rays.  The traversal kernel leaves one hit/miss byte per position.
// The reference's per-fragment `if (result.index < 0)` branches
// (tracer.fs:442,509) are resolved per block: every 256-item tile pushes its hits and its misses into two block-local
// queues and work starts only on full groups of one kind, so hit shading and miss shading never share a warp.
// MAT_TEX: the atlas is the material-interleaved one (false = plain RGBA8 layers, the fallback of fspt_scene_upload);
// a template parameter so that only one of the two sampling routines is in the kernel's instruction footprint.
// LIST (adaptive sampling): path j * S + s belongs to the pixel of slot A.list[j].
template <bool MAT_TEX, bool LIST = false>
__global__ void __launch_bounds__(SHADE_THREADS, SHADE_MIN_BLOCKS) k_shade(const ShadeArgs A) {
  init_unorm8_lut();
  // block-local queues: every tile pushes its hits and misses, and work is only started on FULL groups of
  // SHADE_THREADS items of one kind, so hit shading and miss shading never share a warp (or a block)
  __shared__ int q_hit[2 * SHADE_THREADS], q_miss[2 * SHADE_THREADS];
  __shared__ int s_hits[SHADE_THREADS / 32], s_miss[SHADE_THREADS / 32];
  const int n = A.counts_in[0];
  const unsigned lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
  int nh = 0, nm = 0;  // queue fill, block-uniform
  const int n_tiles = (n + SHADE_THREADS - 1) / SHADE_THREADS;
  // Tiles are handed out by a cursor, so a block that becomes resident late (behind another launch) takes less work
  // instead of a fixed share.  Every block draws tickets until it gets one >= n_tiles, so a launch draws exactly
  // n_tiles + gridDim.x of them; the block that draws the last one puts the cursor back to 0 for the next launch.
  __shared__ int s_tile;
  const unsigned last_ticket = (unsigned)n_tiles + gridDim.x - 1u;
  auto fetch_tile = [&]() {
    const int t = atomicAdd(A.tile_next, 1);
    if ((unsigned)t == last_ticket) atomicExch(A.tile_next, 0);
    s_tile = t;
  };
  if (threadIdx.x == 0) fetch_tile();
  __syncthreads();
  for (;;) {
    const int tile = s_tile;
    const bool last = tile >= n_tiles;  // one extra round drains the partial groups
    if (!last) {
      const int it = tile * SHADE_THREADS + threadIdx.x;
      const bool live = it < n;
      const int slot = it;  // record position
      const bool hit = live && A.hit_flag[it] != 0;  // written by k_trace per position: a coalesced read
      const unsigned mh = __ballot_sync(0xffffffffu, hit), mm = __ballot_sync(0xffffffffu, live && !hit);
      if (lane == 0) { s_hits[warp] = __popc(mh); s_miss[warp] = __popc(mm); }
      __syncthreads();
      if (threadIdx.x == 0) fetch_tile();  // every thread has read s_tile; the next barrier publishes the new one
      int hits_before = 0, miss_before = 0, t_hit = 0, t_miss = 0;
#pragma unroll
      for (int w = 0; w < SHADE_THREADS / 32; ++w) {
        if (w < (int)warp) { hits_before += s_hits[w]; miss_before += s_miss[w]; }
        t_hit += s_hits[w]; t_miss += s_miss[w];
      }
      const unsigned lt = (1u << lane) - 1u;
      if (hit) q_hit[nh + hits_before + __popc(mh & lt)] = slot;
      else if (live) q_miss[nm + miss_before + __popc(mm & lt)] = slot;
      nh += t_hit; nm += t_miss;
      __syncthreads();
    }
    while (nh >= SHADE_THREADS || (last && nh > 0)) {
      const int take = nh < SHADE_THREADS ? nh : SHADE_THREADS;
      bool cont = false, shadow = false;
      PathRecord rec;
      if ((int)threadIdx.x < take) cont = shade_hit<MAT_TEX, LIST>(A, q_hit[nh - take + threadIdx.x], shadow, rec);
      // stream compaction of the surviving paths: the new record goes to the next free position of ps_out
      const int pos_out = append_pos(cont, A.counts_out + 0);
      if (cont) store_record(A.ps_out, pos_out, rec, shadow);
      {
        const int j = append_pos(shadow, A.counts_out + 1);
        if (shadow) {  // origin = the continuation ray's (tracer.fs:501), direction = the sampled environment direction
          float4* sr = A.shadow_rays_out + 2 * (size_t)j;
          sr[0] = make_float4(rec.w[0].x, rec.w[0].y, rec.w[0].z, __int_as_float(pos_out));
          sr[1] = rec.w[2];
        }
      }
      nh -= take;
      __syncthreads();
    }
    while (nm >= SHADE_THREADS || (last && nm > 0)) {
      const int take = nm < SHADE_THREADS ? nm : SHADE_THREADS;
      if ((int)threadIdx.x < take) shade_miss<LIST>(A, q_miss[nm - take + threadIdx.x]);
      nm -= take;
      __syncthreads();
    }
    if (last) break;
  }
}

// ---------------------------------------------------------------------------------------------------------
// tracer.fs:515-517: clamp, then running mean over ticks (mode 0) or plain sum (mode 1), per pixel in tick
// order so that the f32 result equals the reference's sequence of passes.
// sample_color is indexed by the pixel inside the context's rectangle (rw x rh at rx0, ry0), fb by the frame pixel.
// MOMENT (adaptive sampling, adaptive.cuh): the luminance l of every clamped sample adds l*l to *m2, in tick order.
template <bool MOMENT>
__device__ __forceinline__ void accumulate_pixel(const float4* __restrict__ sample_color, float4* fb, float4* last_color,
                                                 int q, size_t p, int n_samples, unsigned first_tick, int mode,
                                                 int sanitize, float* m2) {
  float4 acc = fb[p];
  float m = MOMENT ? m2[p] : 0.0f;
  v3 c = mk3(0.0f, 0.0f, 0.0f);
  for (int s = 0; s < n_samples; ++s) {
    const float4 c4 = sample_color[(size_t)q * n_samples + s];
    c = mk3(c4.x, c4.y, c4.z);
    if (sanitize) {  // deviation from the reference, which lets NaN stick (DESIGN.md section 6)
      if (c.x != c.x) c.x = 0.0f;
      if (c.y != c.y) c.y = 0.0f;
      if (c.z != c.z) c.z = 0.0f;
    }
    c = clamp3(c, 0.0f, 1024.0f);  // :515
    if (MOMENT) {
      const float l = (c.x * 0.2126f + c.y * 0.7152f) + c.z * 0.0722f;
      m += l * l;
    }
    if (mode == 0) {
      const float ft = (float)(first_tick + (unsigned)s);
      const v3 t = mk3(acc.x, acc.y, acc.z);
      const v3 o = div(add(c, mul(t, ft)), ft + 1.0f);  // :517
      acc = make_float4(o.x, o.y, o.z, 1.0f);
    } else {
      acc = make_float4(acc.x + c.x, acc.y + c.y, acc.z + c.z, acc.w + 1.0f);  // alpha = this pixel's sample count
    }
  }
  fb[p] = acc;
  if (MOMENT) m2[p] = m;
  if (last_color) last_color[p] = make_float4(c.x, c.y, c.z, 1.0f);
}
__global__ void __launch_bounds__(256) k_accumulate(const float4* __restrict__ sample_color, float4* fb, float4* last_color,
                                                    int rx0, int ry0, int rw, int rh, int width, int n_samples,
                                                    unsigned first_tick, int mode, int sanitize) {
  const int q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= rw * rh) return;
  const size_t p = (size_t)(ry0 + q / rw) * width + (size_t)(rx0 + q % rw);
  accumulate_pixel<false>(sample_color, fb, last_color, q, p, n_samples, first_tick, mode, sanitize, nullptr);
}

// ---------------------------------------------------------------------------------------------------------
// draw.fs main (:82-93) with filterFireflies (:50-80) and ACESFitted (:39-48), fused: one pass RGBA32F -> RGBA8.
// In sum mode (multi-GPU: sample sets and / or tiles reduced with NCCL) every pixel is divided on the fly by its own
// sample count, which the accumulation kernel keeps in the alpha channel (exact in f32 below 2^24 samples).
__device__ __forceinline__ v3 fb_fetch(const float4* fb, int W, int H, long long cx, long long cy, int use_div) {
  if (cx < 0 || cy < 0 || cx >= W || cy >= H) return mk3(0.0f, 0.0f, 0.0f);  // robust texelFetch
  const float4 v = fb[(size_t)cy * W + (size_t)cx];
  if (use_div) return v.w > 0.0f ? mk3(v.x / v.w, v.y / v.w, v.z / v.w) : mk3(0.0f, 0.0f, 0.0f);
  return mk3(v.x, v.y, v.z);
}
__device__ __forceinline__ float rrt_odt_fit(float v) {  // draw.fs:32-37
  const float a = v * (v + 0.0245786f) - 0.000090537f;
  const float b = v * (0.983729f * v + 0.4329510f) + 0.238081f;
  return a / b;
}
__device__ __forceinline__ unsigned char quant8(float v) {
  if (!(v > 0.0f)) return 0;
  if (v >= 1.0f) return 255;
  return (unsigned char)(int)floorf(v * 255.0f + 0.5f);
}
__global__ void __launch_bounds__(256) k_post(const float4* __restrict__ fb, uchar4* out, int W, int H, float exposure,
                                              float saturation, int denoise, float maxSigma, float scale, int use_div) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y;
  if (x >= W || y >= H) return;
  const v3 lumaCoefs = mk3(0.2126f, 0.7152f, 0.0722f);
  const float fx = (float)x + 0.5f, fy = (float)y + 0.5f;
  const long long bx = coord_to_int(fx * scale), by = coord_to_int(fy * scale);
  v3 texColor;
  if (denoise) {
    float sum = 0.0f, sq_sum = 0.0f;
    v3 middle = mk3(0.0f, 0.0f, 0.0f);
    float middleLuma = 0.0f;
    const float samples = 24.0f;
    for (int i = 0; i < 5; i++)
      for (int j = 0; j < 5; j++) {
        const int osx = i - 2, osy = j - 2;
        const v3 color = fb_fetch(fb, W, H, bx + osx, by + osy, use_div);
        const float luma = dot(color, lumaCoefs);
        if (osx == 0 && osy == 0) { middle = color; middleLuma = luma; continue; }
        sum += luma;
        sq_sum += luma * luma;
      }
    const float mean = sum / samples;
    const float variance = sq_sum / samples - mean * mean;
    const float sigma = sqrtf(variance);
    if (fabsf(middleLuma - mean) > maxSigma * sigma) middle = mul(middle, mean / middleLuma);
    texColor = mul(middle, exposure);
  } else {
    texColor = mul(fb_fetch(fb, W, H, bx, by, use_div), exposure);
  }
  const v3 c = texColor;
  v3 a = mk3(c.x * 0.59719f + c.y * 0.35458f + c.z * 0.04823f, c.x * 0.07600f + c.y * 0.90834f + c.z * 0.01566f,
             c.x * 0.02840f + c.y * 0.13383f + c.z * 0.83777f);
  a = mk3(rrt_odt_fit(a.x), rrt_odt_fit(a.y), rrt_odt_fit(a.z));
  const v3 o = mk3(a.x * 1.60475f + a.y * -0.53108f + a.z * -0.07367f, a.x * -0.10208f + a.y * 1.10813f + a.z * -0.00605f,
                   a.x * -0.00327f + a.y * -0.07276f + a.z * 1.07602f);
  v3 mapped = clamp3(o, 0.0f, 1.0f);
  const float l = dot(mapped, lumaCoefs);
  mapped = mix3(mk3(l, l, l), mapped, saturation);
  mapped = mk3(dm::powf_(mapped.x, 0.454545f), dm::powf_(mapped.y, 0.454545f), dm::powf_(mapped.z, 0.454545f));
  out[(size_t)y * W + x] = make_uchar4(quant8(mapped.x), quant8(mapped.y), quant8(mapped.z), 255);
}

// FSPT-DM2 probes (fspt_debug_math)
__global__ void k_debug_math(int fn, const float* x, const float* y, float* out, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float r = 0.0f;
  switch (fn) {
    case 0: r = dm::sinf_(x[i]); break;
    case 1: r = dm::cosf_(x[i]); break;
    case 2: r = dm::atan2f_(y[i], x[i]); break;
    case 3: r = dm::asinf_(x[i]); break;
    case 4: r = dm::exp2f_(x[i]); break;
    case 5: r = dm::powf_(x[i], y[i]); break;
    case 6: { float s, c; dm::sincosf_(x[i], s, c); r = s; break; }
    case 7: { float s, c; dm::sincosf_(x[i], s, c); r = c; break; }
  }
  out[i] = r;
}
