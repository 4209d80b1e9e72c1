// fspt_api.cu -- context, scene upload (layout repack), wavefront render loop and the extern "C" ABI of
// libfspt_b200.so (include/fspt_b200.h).  Host side of what main.js does between initBVH() and tick():
// texImage uploads (main.js:408-437,548-560,170-180), drawCamera/drawTracer/drawQuad (main.js:741-824).
// Map: Ctx (state of one context) -- stage_atlas (the atlas part of an upload: runs inline or on the context's atlas
// thread) -- launch_trace / render_wave (one wave of the wavefront) -- NCCL loaded at run time, broadcast_phase2 (the
// deferred atlas part of fspt_scene_broadcast) -- extern "C": create / destroy, scene_upload_impl (pre-passes and record
// builders live in scene_pack.h, the worker pool in host_pool.h), render, resolve, accumulation access, debug entry
// points, tiles and collectives, parameters and statistics.
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <nccl.h>  // types only: the library is resolved with dlopen at fspt_comm_init, there is no link-time dependency
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#if defined(__SSE2__)
#include <emmintrin.h>
#endif
#if defined(__SSSE3__)
#include <tmmintrin.h>
#endif
#include <algorithm>
#include <array>
#include <atomic>
#include <map>
#include <memory>
#include <chrono>
#include <condition_variable>
#include <functional>
#include <mutex>
#include <thread>
#include <string>
#include <vector>

#include "../../include/fspt_b200.h"
#include "adaptive.cuh"
#include "device_common.cuh"
#include "host_pool.h"
#include "scene_pack.h"
#include "shade.cuh"
#include "traverse.cuh"

namespace fspt {
thread_local std::string g_create_error;  // fspt_last_error(NULL); the device BVH builder (bvh_device.cu) reports here too
}

namespace {

using fspt::g_create_error;

// A block of device memory (DevBuf) or page-locked host memory (PinnedBuf) that only grows: fit() keeps it when it is
// large enough and re-allocates it otherwise.  Freed on destruction.
template <class T, bool Pinned>
struct GrowBuf {
  T* p = nullptr;
  size_t cap = 0;  // bytes
  GrowBuf() = default;
  GrowBuf(const GrowBuf&) = delete;
  GrowBuf& operator=(const GrowBuf&) = delete;
  ~GrowBuf() { release(); }
  cudaError_t fit(size_t bytes) {
    if (p && cap >= bytes) return cudaSuccess;
    release();
    void* q = nullptr;
    const cudaError_t e = Pinned ? cudaMallocHost(&q, bytes) : cudaMalloc(&q, bytes);
    if (e == cudaSuccess) { p = static_cast<T*>(q); cap = bytes; }
    return e;
  }
  void release() {
    if (p) { if (Pinned) cudaFreeHost(p); else cudaFree(p); }
    p = nullptr; cap = 0;
  }
};
template <class T> using DevBuf = GrowBuf<T, false>;
template <class T> using PinnedBuf = GrowBuf<T, true>;

// A CUDA array (2D when layers == 0, layered otherwise) with its texture object -- point-sampled, clamped, element
// reads -- and, for an array a kernel writes, its surface object.  fit() keeps the array when the format, shape and
// surface flag match and re-creates it otherwise.  Freed on destruction.
struct TexArray {
  cudaArray_t arr = nullptr;
  cudaTextureObject_t tex = 0;
  cudaSurfaceObject_t surf = 0;
  cudaChannelFormatDesc fmt{};
  int w = 0, h = 0, layers = 0;
  bool surface = false;
  TexArray() = default;
  TexArray(const TexArray&) = delete;
  TexArray& operator=(const TexArray&) = delete;
  ~TexArray() { release(); }
  cudaError_t fit(cudaChannelFormatDesc f, int w_, int h_, int layers_, bool surface_) {
    if (arr && !memcmp(&f, &fmt, sizeof f) && w == w_ && h == h_ && layers == layers_ && surface == surface_)
      return cudaSuccess;
    release();
    const unsigned flags = surface_ ? cudaArraySurfaceLoadStore : 0;
    cudaError_t e = layers_ ? cudaMalloc3DArray(&arr, &f, make_cudaExtent(w_, h_, layers_), cudaArrayLayered | flags)
                            : cudaMallocArray(&arr, &f, w_, h_, flags);
    if (e != cudaSuccess) { arr = nullptr; return e; }
    cudaResourceDesc rd = {};
    rd.resType = cudaResourceTypeArray;
    rd.res.array.array = arr;
    cudaTextureDesc td = {};
    td.addressMode[0] = td.addressMode[1] = td.addressMode[2] = cudaAddressModeClamp;
    td.filterMode = cudaFilterModePoint;
    td.readMode = cudaReadModeElementType;
    e = cudaCreateTextureObject(&tex, &rd, &td, nullptr);
    if (e == cudaSuccess && surface_) e = cudaCreateSurfaceObject(&surf, &rd);
    if (e != cudaSuccess) { release(); return e; }
    fmt = f; w = w_; h = h_; layers = layers_; surface = surface_;
    return cudaSuccess;
  }
  void release() {
    if (surf) cudaDestroySurfaceObject(surf);
    if (tex) cudaDestroyTextureObject(tex);
    if (arr) cudaFreeArray(arr);
    arr = nullptr; tex = 0; surf = 0;
    w = h = layers = 0; surface = false;
  }
};

cudaError_t create_handle(cudaStream_t* h, unsigned flags) { return cudaStreamCreateWithFlags(h, flags); }
cudaError_t create_handle(cudaEvent_t* h, unsigned flags) { return cudaEventCreateWithFlags(h, flags); }
void destroy_handle(cudaStream_t h) { cudaStreamDestroy(h); }
void destroy_handle(cudaEvent_t h) { cudaEventDestroy(h); }
void destroy_handle(cudaTextureObject_t h) { cudaDestroyTextureObject(h); }

// A stream, an event (create) or a texture object (created by the caller into `h`), destroyed on destruction or reset.
// Movable, so that a growing std::vector can hold it; converts to the raw handle.
template <class H>
struct Handle {
  H h{};
  Handle() = default;
  Handle(Handle&& o) noexcept : h(o.h) { o.h = H{}; }
  ~Handle() { reset(); }
  cudaError_t create(unsigned flags) {
    reset();
    const cudaError_t e = create_handle(&h, flags);
    if (e != cudaSuccess) h = H{};
    return e;
  }
  void reset() {
    if (h) destroy_handle(h);
    h = H{};
  }
  operator H() const { return h; }
};
using Stream = Handle<cudaStream_t>;
using Event = Handle<cudaEvent_t>;
using TexObject = Handle<cudaTextureObject_t>;

// A resident scene apart from its atlas: what fspt_scene_upload derived from the host buffers and what
// fspt_scene_broadcast sends to the other ranks.  Both size the buffers by it (fit_scene) and make it the scene the
// kernels read (publish_scene).
struct SceneInfo {
  uint64_t bytes_nodes, bytes_tris, bytes_shade, bytes_bins, scene_bytes;
  int32_t root_ref, n_tris, n_interior, atlas_res, atlas_layers, env_w, env_h, n_bins, has_dielectric;
};

// The resident atlas: what stage_atlas made of the caller's layers and what phase 2 of fspt_scene_broadcast sends.
struct AtlasInfo {
  uint64_t bytes_layer_info, bytes_mat_info;
  int32_t interleaved;  // 1: the material-interleaved array (one layer per textured material), 0: the plain RGBA8 array
  int32_t res, layers;
};

// The launch variants of k_trace: plain, with per-slot visit counts (debug), camera-fused (the primary launch of a wave)
// and camera-fused over the listed pixels (adaptive sampling).
enum TraceMode { TRACE_PLAIN, TRACE_COUNT, TRACE_CAMERA, TRACE_CAMERA_LIST, TRACE_MODES };
struct TraceKernel {
  void (*fn)(TraceArgs);
  int blocks = 0;  // persistent grid (fspt_create)
};

// Members are destroyed in reverse order of declaration: the host workers first, a texture object before the buffer it
// reads, the events and streams last.
struct Ctx {
  int device = 0, sm_count = 0;
  int width = 0, height = 0, n_pixels = 0;
  int rx0 = 0, ry0 = 0, rw = 0, rh = 0;  // the pixel rectangle this context renders (fspt_set_tile); default = frame
  static constexpr int RB_SLOTS = 8;    // rand-base staging slots (h_rb)
  static constexpr int POLL_SLOTS = 8;  // refraction poll slots per band (h_poll)

  // streams and events
  Stream stream;
  Stream stream2;      // the second row band of a render (render_wave); forked from and joined to `stream`
  Stream copy_stream;  // atlas DMA, overlaps the primary traversal
  Event ev_fork, ev_join;
  Event ev_begin, ev_end;
  std::vector<Event> ev_trace;  // pairs around traversal (tag 0) / shading (tag 1) launches of the last render
  Event ev_atlas;               // behind the atlas copies (copy_stream) the first shading launch waits for
  Event ev_env;                 // behind the environment copies on the context's stream (recorded when env_in_place)
  std::vector<Event> ev_ring;   // per ring slot (h_ring): the copies that read it have completed
  Event ev_rb[RB_SLOTS];        // per rand-base slot: the copy that read it has completed
  Event ev_poll[2][POLL_SLOTS]; // per band and poll slot (h_poll): the count has landed
  Event ev_red0, ev_red1;       // around the last fspt_reduce_accum
  Event ev_bcast;               // end of phase 1 of fspt_scene_broadcast on the context's stream

  std::vector<int> ev_tag;
  size_t ev_trace_used = 0;
  bool render_timed = false;
  std::string error;

  // scene: buffers and arrays are kept across uploads and reused when they fit
  bool has_scene = false;
  SceneInfo info{};
  AtlasInfo atlas_info{};
  DeviceScene sc{};  // the kernels' view, set by publish_scene / publish_atlas
  DevBuf<uint8_t> d_nodes, d_tris, d_shade, d_bins;
  TexObject nodes_tex;                // the node array again as a linear texture (second L1 data pipe)
  DevBuf<uint2> d_layer_info;
  DevBuf<int4> d_mat_info;
  TexArray env, mat, atlas;           // mat: the material-interleaved atlas; atlas: the plain RGBA8 one (one of the two)
  DevBuf<uint8_t> d_raw;              // distinct varying atlas layers as uploaded (RGBA8), source of the GPU interleave
  DevBuf<uint8_t> d_mat_src;          // MatSrc per textured material
  PinnedBuf<uint8_t> h_stage;         // pinned staging for the atlas (one slot per layer)
  // fspt_scene_upload_async: the atlas part of the upload (constant-layer scan, host interleave into pinned memory,
  // band-wise DMA) runs on this thread after the call has returned; joined before the first shading launch and by
  // everything that touches scene state
  std::thread atlas_thread;
  // page-locked sources are DMA'd in place: they stay borrowed until the copies have completed, not just been enqueued
  bool env_in_place = false, atlas_in_place = false;
  std::atomic<uint64_t> atlas_launches{0};  // kernels launched by the atlas part (folded into stats.kernel_launches)
  int atlas_rc = 0;            // outcome of the atlas part (written by the atlas thread, read after joining it)
  std::string atlas_error;
  PinnedBuf<uint8_t> h_ring;   // pinned ring the geometry records are staged through, chunk by chunk
  PinnedBuf<uint8_t> h_geo;    // pinned block of the small tables (bins, layer / material tables) + env

  // frame state
  DevBuf<float4> d_fb;             // accumulation target (RGBA32F)
  DevBuf<float4> d_last_color;
  DevBuf<float4> d_sample_color;
  DevBuf<float4> d_cam_pos;        // debug_primary only
  DevBuf<float4> d_cam_dir;
  DevBuf<uchar4> d_rgba8;
  uint32_t next_tick = 0;
  uint64_t accum_samples = 0;
  int accum_mode = 0;
  int sanitize = 1;
  int max_refractions = 64;
  int anyhit = 1;
  // adaptive sampling (fspt_set_adaptive), on while adapt_err > 0
  float adapt_err = 0.0f;
  int adapt_min = 2;
  DevBuf<float> d_m2;         // per frame pixel: sum of the squared luminances of its samples (allocated when first on)
  DevBuf<int> d_list;         // slots of the pixels a wave renders: band b's segment starts at its first pixel
  uint64_t adaptive_samples = 0;  // d_stats[8] as last read: path samples of adaptive renders since fspt_clear

  // wavefront state
  int wave_samples = 0;       // samples in flight per wave (whole frame)
  int wave_cap = 64;
  size_t wave_paths = 0;
  PathState ps{};             // = ps2[0] (debug entry points)
  PathState ps2[2]{};         // dense path-record arrays, ping-pong: shade reads one, compacts survivors into the other
  DevBuf<float4> d_rec[2];    // what ps2[k] points to
  DevBuf<unsigned char> d_sh[2];
  DevBuf<float4> d_shadow;    // shadow rays of the current bounce, dense: origin | record position, direction | -
  // per band b, from b * BAND_INTS: set k at [2k, 2k+1] = (#continuation, #shadow), [8] active pixels of the wave
  // (adaptive sampling), [32] traversal fetch cursor, [64] shading tile cursor -- each cursor on a 128-byte line of its
  // own: every warp's (block's) atomicAdd hits it
  static constexpr int BAND_INTS = 96;
  DevBuf<int> d_counts;
  DevBuf<int> d_count_out;    // per-slot visit count (debug)
  DevBuf<unsigned char> d_hit_flag;  // hit / miss per record position
  DevBuf<unsigned long long> d_stats;  // rays, nodes, leaves, capped
  DevBuf<float> d_rb;         // rand bases of one render call: [0,cap) camera, [cap,2cap) tracer
  // pinned staging, a ring of RB_SLOTS blocks of 2*rb_cap floats: a slot is rewritten only after the copy that last
  // read it has completed (ev_rb), so fspt_render never waits for the GPU to drain
  PinnedBuf<float> h_rb;
  int rb_slot = 0;
  int rb_cap = 0;
  // refraction bounces beyond NUM_BOUNCES (tracer.fs:488): path counts polled two iterations behind the enqueue
  PinnedBuf<int> h_poll;                   // [band * POLL_SLOTS + slot], each behind its event ev_poll[band][slot]
  // collectives (fspt_comm_init): NCCL communicator over NVLink / NVSwitch
  ncclComm_t comm = nullptr;
  int comm_rank = 0, comm_world = 1;
  bool reduce_timed = false;
  DevBuf<uint8_t> d_lin;      // linear staging of the atlas array for fspt_scene_broadcast (phase 2)
  DevBuf<uint8_t> d_hdr;      // broadcast headers
  DevBuf<uint8_t> d_lin_env;  // linear staging of the environment array (phase 1 of the broadcast)
  int bcast_pending_root = -1;  // >= 0: phase 2 of fspt_scene_broadcast (the atlas) has not been issued yet
  // the kernel variants: k_trace by [TraceMode][node texture; 0: the node array is beyond the linear-texture limit],
  // each with its persistent grid, and k_shade by [mat_tex][list], all with the grid of k_shade<true>
  TraceKernel trace_kernels[TRACE_MODES][2] = {
      {{k_trace<false, false, false>}, {k_trace<false, false, true>}},
      {{k_trace<true, false, false>}, {k_trace<true, false, true>}},
      {{k_trace<false, true, false>}, {k_trace<false, true, true>}},
      {{k_trace<false, true, false, true>}, {k_trace<false, true, true, true>}},
  };
  void (*shade_kernels[2][2])(ShadeArgs) = {{k_shade<false>, k_shade<false, true>}, {k_shade<true>, k_shade<true, true>}};
  int shade_blocks = 0;

  fspt_stats stats{};
  std::unique_ptr<HostPool> pool;  // host workers of fspt_scene_upload (created at the first upload)
};

void comm_free(Ctx* c);
int broadcast_phase2(Ctx* c);

int fail(Ctx* c, int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  if (c) c->error = buf; else g_create_error = buf;
  return code;
}

// CK_INTO: the message of a failed call goes to `dst` (stage_atlas reports into atlas_error: it runs on the atlas thread
// while the caller may write c->error)
#define CK_INTO(dst, call)                                                                  \
  do {                                                                                      \
    cudaError_t e_ = (call);                                                                \
    if (e_ != cudaSuccess) {                                                                \
      (dst) = std::string(#call) + " failed: " + cudaGetErrorString(e_);                    \
      return FSPT_E_CUDA;                                                                   \
    }                                                                                       \
  } while (0)
#define CK(call) CK_INTO(c->error, call)

// A device array of 16-byte words as a linear texture (tex1Dfetch): the second L1 data path next to the LSU.  Arrays
// beyond the 2^27-texel limit get no texture (0) and are read with plain loads.
int linear_tex(Ctx* c, TexObject* tex, void* ptr, size_t bytes, bool allowed) {
  tex->reset();
  if (!allowed || bytes / 16 > ((size_t)1 << 27) || bytes == 0) return FSPT_OK;
  cudaResourceDesc r = {};
  r.resType = cudaResourceTypeLinear;
  r.res.linear.devPtr = ptr;
  r.res.linear.desc = cudaCreateChannelDesc<float4>();
  r.res.linear.sizeInBytes = bytes;
  cudaTextureDesc t = {};
  t.readMode = cudaReadModeElementType;
  CK(cudaCreateTextureObject(&tex->h, &r, &t, nullptr));
  return FSPT_OK;
}

// Storage for the scene `s` (reused when it fits): the geometry records, the bins and the environment array.
int fit_scene(Ctx* c, const SceneInfo& s) {
  CK(c->d_nodes.fit(s.bytes_nodes));
  CK(c->d_tris.fit(s.bytes_tris));
  CK(c->d_shade.fit(s.bytes_shade));
  CK(c->d_bins.fit(s.bytes_bins));
  CK(c->env.fit(cudaCreateChannelDesc<uchar4>(), s.env_w, s.env_h, 0, false));  // RGBA8 RGBE (main.js:170-180)
  return FSPT_OK;
}

// Makes `s`, in the storage of fit_scene, the scene the kernels read (the atlas part: publish_atlas).
int publish_scene(Ctx* c, const SceneInfo& s) {
  // FSPT_NO_NODE_TEX: test knob for the LSU-only instantiation of k_trace
  if (int rc = linear_tex(c, &c->nodes_tex, c->d_nodes.p, s.bytes_nodes, !getenv("FSPT_NO_NODE_TEX"))) return rc;
  c->info = s;
  DeviceScene& sc = c->sc;
  sc.nodes = reinterpret_cast<const float4*>(c->d_nodes.p);
  sc.tris = reinterpret_cast<const float4*>(c->d_tris.p);
  sc.shade = reinterpret_cast<const float4*>(c->d_shade.p);
  sc.bins = reinterpret_cast<const float4*>(c->d_bins.p);
  sc.env = c->env.tex;
  sc.root_ref = s.root_ref;
  sc.n_tris = s.n_tris; sc.n_interior = s.n_interior;
  sc.atlas_res = s.atlas_res; sc.atlas_layers = s.atlas_layers; sc.env_w = s.env_w; sc.env_h = s.env_h;
  sc.n_bins = s.n_bins;
  set_env_constants(sc);
  return FSPT_OK;
}

// Makes one form of the atlas resident, `res` x `res` x `layers`, and frees the other: the material-interleaved array
// (uint4 texels) or the plain RGBA8 one.
cudaError_t fit_atlas(Ctx* c, bool interleaved, int res, int layers, bool surface) {
  (interleaved ? c->atlas : c->mat).release();
  return interleaved ? c->mat.fit(cudaCreateChannelDesc<uint4>(), res, res, layers, surface)
                     : c->atlas.fit(cudaCreateChannelDesc<uchar4>(), res, res, layers, surface);
}

// Makes the resident atlas and its two tables the ones k_shade reads.
void publish_atlas(Ctx* c, const AtlasInfo& a) {
  c->atlas_info = a;
  c->sc.mat_tex = c->mat.tex;
  c->sc.atlas = c->atlas.tex;
  c->sc.layer_info = c->d_layer_info.p;
  c->sc.mat_info = c->d_mat_info.p;
}

int alloc_wave(Ctx* c) {
  // samples in flight: traversal launches amortise their ramp/tail over tens of millions of rays (measured at
  // 1280x720: 4 -> 16 -> 32 -> 64 samples per wave = +14 % -> +3 % -> +2.7 %); 64 M paths x (2 x 80 B records + lists)
  // = ~14 GB of 180 GB
  const size_t target_paths = (size_t)64 << 20;
  int S = (int)std::max<size_t>(1, target_paths / (size_t)c->n_pixels);
  S = std::min(S, 64);
  c->wave_cap = 64;
  if (const char* e = getenv("FSPT_WAVE_SAMPLES")) c->wave_cap = S = std::max(1, std::min(64, atoi(e)));  // tuning knob
  c->wave_samples = S;
  c->wave_paths = (size_t)S * c->n_pixels;
  const size_t W = c->wave_paths;
  for (int k = 0; k < 2; ++k) {
    CK(c->d_rec[k].fit(W * 16 * FSPT_PATH_WORDS));
    CK(c->d_sh[k].fit(W));
    c->ps2[k].rec = c->d_rec[k].p;
    c->ps2[k].sh = c->d_sh[k].p;
  }
  c->ps = c->ps2[0];
  CK(c->d_shadow.fit(W * 32));
  CK(c->d_counts.fit(2 * Ctx::BAND_INTS * sizeof(int)));
  CK(cudaMemset(c->d_counts.p, 0, 2 * Ctx::BAND_INTS * sizeof(int)));
  CK(c->d_count_out.fit(W * sizeof(int)));
  CK(c->d_hit_flag.fit(W));
  // [0..3] live, [4..7] snapshot at render start, [8] path samples of adaptive renders since fspt_clear
  CK(c->d_stats.fit(9 * sizeof(unsigned long long)));
  CK(cudaMemset(c->d_stats.p, 0, 9 * sizeof(unsigned long long)));
  CK(c->d_sample_color.fit(W * 16));
  c->rb_cap = 64;
  CK(c->d_rb.fit(2 * (size_t)c->rb_cap * sizeof(float)));
  CK(c->h_rb.fit(Ctx::RB_SLOTS * 2 * (size_t)c->rb_cap * sizeof(float)));
  for (Event& e : c->ev_rb) CK(e.create(cudaEventDisableTiming));
  CK(c->h_poll.fit(2 * Ctx::POLL_SLOTS * sizeof(int)));
  for (auto& band : c->ev_poll)
    for (Event& e : band) CK(e.create(cudaEventDisableTiming));
  return FSPT_OK;
}

// ---- traversal launch helpers ---------------------------------------------------------------------------
// Band b of a render (render_wave) runs on its own stream and has its own counts and cursors; band 0 is the context's
// stream, which every other entry point uses.
cudaStream_t band_stream(const Ctx* c, int band) { return band ? c->stream2 : c->stream; }
int* band_counts(const Ctx* c, int band) { return c->d_counts.p + Ctx::BAND_INTS * band; }

int record_trace_begin(Ctx* c, cudaStream_t s, int tag) {
  while (c->ev_trace_used + 2 > c->ev_trace.size()) {
    Event e;
    CK(e.create(cudaEventDefault));
    c->ev_trace.push_back(std::move(e));
  }
  if (c->ev_tag.size() < c->ev_trace.size() / 2) c->ev_tag.resize(c->ev_trace.size() / 2);
  c->ev_tag[c->ev_trace_used / 2] = tag;
  cudaEventRecord(c->ev_trace[c->ev_trace_used], s);
  return FSPT_OK;
}
void record_trace_end(Ctx* c, cudaStream_t s) {
  cudaEventRecord(c->ev_trace[c->ev_trace_used + 1], s);
  c->ev_trace_used += 2;
}

// One texel of a material layer = the RGBA8 texels of its four maps (device_common.cuh "MatTexel"), each taken from an
// uploaded raw layer or, for a colour layer, from its constant.
struct MatSrc { int raw[4]; unsigned cst[4]; };
// RGB24: the raw layers travelled without their alpha channel (3 bytes per texel) -- tracer.fs:453-456 reads .rgb / .rg of
// the four maps, never .a, so alpha cannot influence an image and is not worth a quarter of the PCIe time.
template <bool RGB24>
__global__ void __launch_bounds__(256) k_interleave_atlas(cudaSurfaceObject_t surf, const uint8_t* __restrict__ raw,
                                                          const MatSrc* __restrict__ src, int R, size_t layer_texels) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y;
  if (x >= R || y >= R) return;
  const MatSrc m = src[blockIdx.z];
  const size_t i = (size_t)y * R + x;
  auto fetch = [&](int k) -> unsigned {
    if (m.raw[k] < 0) return m.cst[k];
    if (RGB24) {
      const uint8_t* p = raw + ((size_t)m.raw[k] * layer_texels + i) * 3;
      return (unsigned)p[0] | ((unsigned)p[1] << 8) | ((unsigned)p[2] << 16);
    }
    return reinterpret_cast<const uint32_t*>(raw)[(size_t)m.raw[k] * layer_texels + i];
  };
  uint4 v;
  v.x = fetch(0); v.y = fetch(1); v.z = fetch(2); v.w = fetch(3);
  surf2DLayeredwrite(v, surf, x * 16, y, blockIdx.z);
}

// counts = band_counts().  The shading tile cursor [64] is zeroed here at the start of every wave; between the shading
// launches of a wave, k_shade puts it back to 0 itself (the block that draws a launch's last ticket), which holds as long
// as every launch runs to completion with the grid it was launched with.  per_active > 0 (adaptive sampling): n_cont is
// per_active paths for each active pixel k_select_active counted into [8].
__global__ void k_set_counts(int* counts, int n_cont, int n_shadow, int per_active) {
  if (per_active) n_cont = per_active * counts[8];
  counts[0] = n_cont; counts[1] = n_shadow; counts[2] = 0; counts[3] = 0; counts[32] = 0; counts[64] = 0;
}

// true when `p` points into page-locked host memory (cudaHostRegister / cudaMallocHost, by whoever): DMA can read it in place
bool host_is_pinned(const void* p) {
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { (void)cudaGetLastError(); return false; }
  return a.type == cudaMemoryTypeHost;
}

// Page-locked sources (fspt_host_register) are read by the copy engines where they lie: the caller gets them back when
// those copies have completed.  (Staged sources were copied out before the upload returned / the atlas thread ended.)
int release_borrowed(Ctx* c) {
  if (c->env_in_place) { CK(cudaEventSynchronize(c->ev_env)); c->env_in_place = false; }
  if (c->atlas_in_place) { CK(cudaEventSynchronize(c->ev_atlas)); c->atlas_in_place = false; }
  return FSPT_OK;
}

// Waits for the atlas part of the last fspt_scene_upload_async (no-op otherwise) and reports its outcome.
int atlas_join(Ctx* c) {
  if (c->atlas_thread.joinable()) c->atlas_thread.join();
  const int rc = c->atlas_rc;
  c->atlas_rc = FSPT_OK;
  if (rc) { c->has_scene = false; c->error = "atlas upload: " + c->atlas_error; }
  return rc;
}

// ---- the atlas part of a scene upload (main.js:548-560) ------------------------------------------------------
// Constant-colour layers are detected (exact: every texel compared), then the atlas is re-interleaved per material into
// 16-byte texels (device_common.cuh "MatTexel") in pinned memory by the host workers and DMA'd band by band as the bands
// land; a scene with so many layer combinations that this would not fit falls back to the plain RGBA8 layered array.
// Everything travels on the copy stream and ends with ev_atlas: only k_shade reads what this function uploads, so a
// render's camera + primary traversal launch overlaps it.  Runs inline (fspt_scene_upload) or on the context's atlas
// thread (fspt_scene_upload_async); every input is held by value or lives in the context's pinned blocks.
struct AtlasJob {
  const uint8_t* atlas;                     // caller's layers, RGBA8, L x R x R
  int L, R;
  std::vector<std::array<int, 4>> mats;     // distinct layer quadruples (diffuse, emission, metallic-roughness, normal)
  uint32_t* layer_info;                     // pinned: per layer {constant?, first texel}
  int32_t* mat_info;                        // pinned: per material 2 x int4
  size_t n_mat_info;                        // ints
  MatSrc* mat_src;                          // pinned: per textured material (GPU-side interleave)
  std::vector<uint8_t> varied;               // per layer: 1 = not a constant colour (scanned next to the geometry staging);
                                             // empty: the atlas part scans the layers itself
  bool src_pinned;                           // the caller's atlas is page-locked (fspt_host_register): no staging copy
  int workers;
  bool timing;
};

// constant-colour layers: constant <=> every texel equals its successor (exact: every texel compared); work item =
// (layer, band), abandoned once the layer is known to vary
constexpr int SCAN_BANDS = 8;
inline void scan_layer_band(const uint8_t* atlas, size_t layer_texels, int item, std::atomic<int>* varied) {
  const int l = item / SCAN_BANDS, band = item % SCAN_BANDS;
  if (varied[l].load(std::memory_order_relaxed)) return;
  const uint32_t* px = reinterpret_cast<const uint32_t*>(atlas) + (size_t)l * layer_texels;
  const size_t i0 = layer_texels * band / SCAN_BANDS, i1 = std::min(layer_texels - 1, layer_texels * (band + 1) / SCAN_BANDS);
  for (size_t i = i0; i < i1;) {
    const size_t n = std::min<size_t>(i1 - i, 16384);
    if (memcmp(px + i, px + i + 1, n * 4) != 0) { varied[l].store(1, std::memory_order_relaxed); return; }
    i += n;
  }
}

int stage_atlas(Ctx* c, const AtlasJob& J) {
  std::string& err = c->atlas_error;
  auto t_prev = std::chrono::steady_clock::now();
  auto lap = [&](const char* what) {
    if (!J.timing) return;
    auto now = std::chrono::steady_clock::now();
    fprintf(stderr, "[fspt upload]   atlas: %-24s %7.2f ms\n", what, std::chrono::duration<double, std::milli>(now - t_prev).count());
    t_prev = now;
  };
  const int L = J.L, R = J.R;
  const size_t layer_texels = (size_t)R * R, layer_bytes = layer_texels * 4;
  const std::vector<std::array<int, 4>>& mats = J.mats;
  uint32_t* layer_info = J.layer_info;
  int32_t* mat_info = J.mat_info;
  HostPool& pool = *c->pool;
  {
    std::vector<std::atomic<int>> varied((size_t)L);
    if (J.varied.empty()) {
      for (auto& v : varied) v.store(0);
      pool.run(L * SCAN_BANDS, J.workers, [&](int item) { scan_layer_band(J.atlas, layer_texels, item, varied.data()); });
      lap("constant-layer scan");
    }
    for (int l = 0; l < L; ++l) {
      layer_info[2 * l] = (J.varied.empty() ? varied[l].load() : J.varied[l]) ? 0u : 1u;
      memcpy(&layer_info[2 * l + 1], J.atlas + (size_t)l * layer_bytes, 4);
    }
  }
  memset(mat_info, 0, J.n_mat_info * 4);
  int n_tex_mats = 0;
  for (size_t m = 0; m < mats.size(); ++m) {
    bool all_const = true;
    for (int k = 0; k < 4; ++k) all_const = all_const && layer_info[2 * mats[m][k]];
    mat_info[8 * m] = all_const ? -1 : n_tex_mats++;
    for (int k = 0; k < 4; ++k) mat_info[8 * m + 1 + k] = (int32_t)layer_info[2 * mats[m][k] + 1];
  }
  // The interleaved atlas costs res^2 * 16 bytes per TEXTURED MATERIAL (distinct layer quadruple) and the same again in
  // pinned staging; quadruples can outnumber layers, so it is bounded against the plain atlas (4 x its bytes, at least
  // 256 MB) and against the free device memory, and any allocation failure falls back to the plain RGBA8 array.
  bool use_mat_tex = !getenv("FSPT_PLAIN_ATLAS");
  const int ML = std::max(1, n_tex_mats);  // layers of the interleaved array
  {
    const size_t inter = (size_t)n_tex_mats * layer_texels * 16, plain = (size_t)L * layer_bytes;
    // the array of the previous upload is reused when it has the same shape: then nothing is allocated and the driver is
    // not asked for the free memory (cudaMemGetInfo is a resource-manager call: usually 0.1 ms, but 20-100 ms every few
    // dozen calls on the virtualised hosts measured, which showed up as spikes in the end-to-end step time)
    const TexArray& mat = c->mat;
    const bool reuse = mat.arr && mat.w == R && mat.layers == ML;
    size_t free_b = (size_t)48 << 30, total_b = 0;
    if (!reuse && cudaMemGetInfo(&free_b, &total_b) != cudaSuccess) { (void)cudaGetLastError(); free_b = (size_t)48 << 30; }
    const size_t resident = (size_t)mat.w * mat.h * 16 * (size_t)mat.layers;  // freed before the new one
    if (inter > std::max<size_t>(4 * plain, (size_t)256 << 20) || inter > ((size_t)48 << 30) ||
        (!reuse && inter > (free_b + resident) / 2))
      use_mat_tex = false;
    if (getenv("FSPT_FORCE_MAT_TEX")) use_mat_tex = true;  // test knob: exercise the allocation-failure fallback
  }
  lap("tables + sizing");
  std::atomic<int> cuda_err(0);
  std::mutex mu;  // serialises the enqueues of the staging items
  bool plain_atlas = !use_mat_tex;
  if (use_mat_tex) {
    // Where the interleave runs.  On the host (default): the 16-byte texels are built in pinned memory and DMA'd.  On the
    // GPU: only the DISTINCT varying layers cross PCIe as raw RGBA8 and k_interleave_atlas builds the texels through a
    // surface -- a material with one image map and three colours then costs 1 layer of staging and DMA instead of 4.
    // Measured break-even (bench scene, 7 varying layers behind 2 materials: GPU path 20 % slower): chosen when the raw
    // layers are at most half of the interleaved bytes.  FSPT_ATLAS_INTERLEAVE=gpu|cpu overrides.
    std::vector<int> raw_of((size_t)L, -1), raw_layers;
    MatSrc* mat_src = J.mat_src;
    for (size_t m = 0; m < mats.size(); ++m) {
      const int tl = mat_info[8 * m];
      if (tl < 0) continue;
      for (int k = 0; k < 4; ++k) {
        const int l = mats[m][k];
        if (!layer_info[2 * l] && raw_of[l] < 0) { raw_of[l] = (int)raw_layers.size(); raw_layers.push_back(l); }
        mat_src[tl].raw[k] = layer_info[2 * l] ? -1 : raw_of[l];
        mat_src[tl].cst[k] = layer_info[2 * l + 1];
      }
    }
    // A page-locked source (the host registered its atlas, fspt_host_register) needs no staging at all on the GPU path:
    // the distinct varying layers are DMA'd from where they lie, the host does nothing but enqueue the copies.
    bool gpu_interleave = n_tex_mats > 0 && (J.src_pinned || raw_layers.size() * 2 <= (size_t)n_tex_mats * 4);
    if (const char* e = getenv("FSPT_ATLAS_INTERLEAVE")) gpu_interleave = n_tex_mats > 0 && !strcmp(e, "gpu");
    const bool direct = gpu_interleave && J.src_pinned;
    c->atlas_in_place = direct;
    // wire format of the staged GPU path: RGB, 3 bytes per texel (the shaders never read alpha, tracer.fs:453-456); the
    // direct path copies the RGBA8 layers as they lie
    const size_t wire_layer_bytes = direct ? layer_bytes : layer_texels * 3;
    const size_t max_ml = getenv("FSPT_FORCE_MAT_TEX") ? (size_t)atoi(getenv("FSPT_FORCE_MAT_TEX")) : (size_t)1 << 30;
    if ((size_t)ML > max_ml ||  // (test knob: pretend the device cannot hold more than that many material layers)
        fit_atlas(c, true, R, ML, gpu_interleave) != cudaSuccess) {
      (void)cudaGetLastError();
      plain_atlas = true;
    }
    const size_t need = gpu_interleave ? wire_layer_bytes * raw_layers.size() : layer_texels * 16 * (size_t)ML;
    if (!plain_atlas && !direct && c->h_stage.fit(need) != cudaSuccess) {
      (void)cudaGetLastError();
      plain_atlas = true;
    }
    lap("arrays + pinned block");
    if (plain_atlas) {
      // could not hold the interleaved atlas: every material becomes "plain" (the tables are not consulted by k_shade<false>)
    } else if (gpu_interleave) {
      CK_INTO(err, c->d_raw.fit(need));
      CK_INTO(err, c->d_mat_src.fit(sizeof(MatSrc) * (size_t)ML));
      if (direct) {
        for (size_t ri = 0; ri < raw_layers.size(); ++ri)
          CK_INTO(err, cudaMemcpyAsync(c->d_raw.p + ri * layer_bytes, J.atlas + (size_t)raw_layers[ri] * layer_bytes,
                                       layer_bytes, cudaMemcpyHostToDevice, c->copy_stream));
      }
      // work item = (raw layer, band of rows): drop the alpha channel into the pinned block, DMA the band
      const int bands = std::max(1, std::min(R, 16));
      pool.run(direct ? 0 : (int)raw_layers.size() * bands, J.workers, [&](int item) {
        const int ri = item / bands, band = item % bands;
        const size_t y0 = (size_t)R * band / bands, y1 = (size_t)R * (band + 1) / bands;
        const size_t off = (size_t)ri * wire_layer_bytes + y0 * R * 3, bytes = (y1 - y0) * R * 3;
        const uint8_t* src = J.atlas + (size_t)raw_layers[ri] * layer_bytes + y0 * R * 4;
        uint8_t* dst = c->h_stage.p + off;
        const size_t n = (y1 - y0) * R;
        size_t i = 0;
#if defined(__SSSE3__)
        // 4 texels (16 bytes) -> 12 bytes per shuffle; the 16-byte store's last 4 bytes are overwritten by the next one
        const __m128i sh = _mm_setr_epi8(0, 1, 2, 4, 5, 6, 8, 9, 10, 12, 13, 14, -1, -1, -1, -1);
        for (; i + 8 <= n; i += 4)
          _mm_storeu_si128(reinterpret_cast<__m128i*>(dst + 3 * i),
                           _mm_shuffle_epi8(_mm_loadu_si128(reinterpret_cast<const __m128i*>(src + 4 * i)), sh));
#endif
        for (; i < n; ++i) { dst[3 * i] = src[4 * i]; dst[3 * i + 1] = src[4 * i + 1]; dst[3 * i + 2] = src[4 * i + 2]; }
        std::lock_guard<std::mutex> g(mu);
        cudaError_t e = cudaMemcpyAsync(c->d_raw.p + off, c->h_stage.p + off, bytes, cudaMemcpyHostToDevice, c->copy_stream);
        if (e != cudaSuccess) cuda_err.store((int)e);
      });
      CK_INTO(err, cudaMemcpyAsync(c->d_mat_src.p, mat_src, sizeof(MatSrc) * (size_t)n_tex_mats, cudaMemcpyHostToDevice, c->copy_stream));
      const dim3 blk(32, 8), grd((R + 31) / 32, (R + 7) / 8, n_tex_mats);
      if (!direct)
        k_interleave_atlas<true><<<grd, blk, 0, c->copy_stream>>>(c->mat.surf, c->d_raw.p,
                                                                  reinterpret_cast<const MatSrc*>(c->d_mat_src.p), R, layer_texels);
      else
        k_interleave_atlas<false><<<grd, blk, 0, c->copy_stream>>>(c->mat.surf, c->d_raw.p,
                                                                   reinterpret_cast<const MatSrc*>(c->d_mat_src.p), R, layer_texels);
      c->atlas_launches.fetch_add(1);
      CK_INTO(err, cudaGetLastError());
    } else {
      // work item = (textured material, band of rows): interleave the four source layers, DMA the band
      const int bands = std::max(1, std::min(R, 16));
      std::vector<int> tex_mat_ids;
      for (size_t m = 0; m < mats.size(); ++m) if (mat_info[8 * m] >= 0) tex_mat_ids.push_back((int)m);
      pool.run((int)tex_mat_ids.size() * bands, J.workers, [&](int item) {
        const int m = tex_mat_ids[item / bands], band = item % bands;
        const int tl = mat_info[8 * m];
        const int y0 = (int)((long long)R * band / bands), y1 = (int)((long long)R * (band + 1) / bands);
        const uint32_t* src[4];
        for (int k = 0; k < 4; ++k) src[k] = reinterpret_cast<const uint32_t*>(J.atlas) + (size_t)mats[m][k] * layer_texels;
        uint32_t* dst = reinterpret_cast<uint32_t*>(c->h_stage.p) + ((size_t)tl * layer_texels + (size_t)y0 * R) * 4;
        const size_t i0 = (size_t)y0 * R, n = (size_t)(y1 - y0) * R;
        size_t i = 0;
#if defined(__SSE2__)
        // 4x4 transpose of 32-bit texels, written with non-temporal stores: the staging block is only read by the DMA
        // engine, so it should neither be fetched for ownership nor displace the source layers from the CPU caches
        for (; i + 4 <= n; i += 4) {
          const __m128i a = _mm_loadu_si128(reinterpret_cast<const __m128i*>(src[0] + i0 + i));
          const __m128i b = _mm_loadu_si128(reinterpret_cast<const __m128i*>(src[1] + i0 + i));
          const __m128i c2 = _mm_loadu_si128(reinterpret_cast<const __m128i*>(src[2] + i0 + i));
          const __m128i d = _mm_loadu_si128(reinterpret_cast<const __m128i*>(src[3] + i0 + i));
          const __m128i ab_lo = _mm_unpacklo_epi32(a, b), ab_hi = _mm_unpackhi_epi32(a, b);
          const __m128i cd_lo = _mm_unpacklo_epi32(c2, d), cd_hi = _mm_unpackhi_epi32(c2, d);
          __m128i* o = reinterpret_cast<__m128i*>(dst + 4 * i);  // 16-byte aligned: pinned block + multiples of 16
          _mm_stream_si128(o + 0, _mm_unpacklo_epi64(ab_lo, cd_lo));
          _mm_stream_si128(o + 1, _mm_unpackhi_epi64(ab_lo, cd_lo));
          _mm_stream_si128(o + 2, _mm_unpacklo_epi64(ab_hi, cd_hi));
          _mm_stream_si128(o + 3, _mm_unpackhi_epi64(ab_hi, cd_hi));
        }
        _mm_sfence();
#endif
        for (; i < n; ++i) {
          dst[4 * i + 0] = src[0][i0 + i]; dst[4 * i + 1] = src[1][i0 + i];
          dst[4 * i + 2] = src[2][i0 + i]; dst[4 * i + 3] = src[3][i0 + i];
        }
        cudaMemcpy3DParms cp = {};
        cp.srcPtr = make_cudaPitchedPtr(dst, (size_t)R * 16, R, y1 - y0);
        cp.dstArray = c->mat.arr;
        cp.dstPos = make_cudaPos(0, y0, tl);
        cp.extent = make_cudaExtent(R, y1 - y0, 1);
        cp.kind = cudaMemcpyHostToDevice;
        std::lock_guard<std::mutex> g(mu);
        cudaError_t e = cudaMemcpy3DAsync(&cp, c->copy_stream);
        if (e != cudaSuccess) cuda_err.store((int)e);
      });
    }
  }
  if (plain_atlas) {
    CK_INTO(err, fit_atlas(c, false, R, L, false));
    CK_INTO(err, c->h_stage.fit(layer_bytes * L));
    pool.run(L, J.workers, [&](int l) {
      uint8_t* dst = c->h_stage.p + (size_t)l * layer_bytes;
      memcpy(dst, J.atlas + (size_t)l * layer_bytes, layer_bytes);
      cudaMemcpy3DParms cp = {};
      cp.srcPtr = make_cudaPitchedPtr(dst, (size_t)R * 4, R, R);
      cp.dstArray = c->atlas.arr;
      cp.dstPos = make_cudaPos(0, 0, l);
      cp.extent = make_cudaExtent(R, R, 1);
      cp.kind = cudaMemcpyHostToDevice;
      std::lock_guard<std::mutex> g(mu);
      cudaError_t e = cudaMemcpy3DAsync(&cp, c->copy_stream);
      if (e != cudaSuccess) cuda_err.store((int)e);
    });
  }
  if (cuda_err.load()) {
    err = std::string("a staging copy failed: ") + cudaGetErrorString((cudaError_t)cuda_err.load());
    return FSPT_E_CUDA;
  }
  lap("stage + enqueue");
  // the two small tables k_shade reads next to the texels: same stream, so the same event covers them
  const AtlasInfo a = {(uint64_t)L * 8, J.n_mat_info * 4, !plain_atlas, R, plain_atlas ? L : ML};
  CK_INTO(err, c->d_layer_info.fit(a.bytes_layer_info));
  CK_INTO(err, c->d_mat_info.fit(a.bytes_mat_info));
  CK_INTO(err, cudaMemcpyAsync(c->d_layer_info.p, layer_info, a.bytes_layer_info, cudaMemcpyHostToDevice, c->copy_stream));
  CK_INTO(err, cudaMemcpyAsync(c->d_mat_info.p, mat_info, a.bytes_mat_info, cudaMemcpyHostToDevice, c->copy_stream));
  publish_atlas(c, a);
  CK_INTO(err, cudaEventRecord(c->ev_atlas, c->copy_stream));
  return FSPT_OK;
}

// The path records, shadow rays, hit flags and sample colours of a band: its slice of the wave's arrays, from path `off`.
struct BandSlice {
  PathState ps[2];
  float4* shadow;
  unsigned char* hit_flag;
  float4* sample_color;
};
BandSlice band_slice(const Ctx* c, size_t off) {
  BandSlice b;
  for (int k = 0; k < 2; ++k) {
    b.ps[k].rec = c->ps2[k].rec + FSPT_PATH_WORDS * off;
    b.ps[k].sh = c->ps2[k].sh + off;
  }
  b.shadow = c->d_shadow.p + 2 * off;
  b.hit_flag = c->d_hit_flag.p + off;
  b.sample_color = c->d_sample_color.p + off;
  return b;
}

// Traverses the continuation ray of every record of array `which` (counts[2*which] of them) + counts[2*which+1]
// shadow rays of band `band` (slice `sl`); results go into the records, plus one hit/miss byte per position (for k_shade).
int launch_trace(Ctx* c, int band, const BandSlice& sl, int which, bool hit_flags, bool write_count,
                 const FrameParams* cam = nullptr, const float* rb_cam = nullptr, int n_samples = 1,
                 const int* list = nullptr) {
  TraceArgs A;
  if (cam) A.f = *cam; else memset(&A.f, 0, sizeof A.f);
  A.rb_cam = rb_cam; A.n_samples = n_samples;
  A.div_s = make_fastdiv((unsigned)std::max(1, n_samples), c->wave_paths);
  A.anyhit = c->anyhit;
  A.nodes = c->sc.nodes; A.tris = c->sc.tris; A.root_ref = c->sc.root_ref; A.nodes_tex = c->nodes_tex;
  A.ps = sl.ps[which];
  A.shadow_rays = sl.shadow;
  A.counts = band_counts(c, band) + 2 * which;
  A.next = band_counts(c, band) + 32;
  A.stats = c->d_stats.p;
  A.count_out = write_count ? c->d_count_out.p : nullptr;
  A.hit_flag = hit_flags ? sl.hit_flag : nullptr;
  A.list = list;
  const cudaStream_t s = band_stream(c, band);
  // (a pixel list comes with camera-fused launches only)
  const int mode = list ? TRACE_CAMERA_LIST : cam ? TRACE_CAMERA : write_count ? TRACE_COUNT : TRACE_PLAIN;
  const TraceKernel& k = c->trace_kernels[mode][A.nodes_tex != 0];
  if (int rc = record_trace_begin(c, s, cam ? 2 : 0)) return rc;  // tag 2: the camera-fused primary launch of a wave
  k.fn<<<k.blocks, TRACE_THREADS, 0, s>>>(A);
  record_trace_end(c, s);
  c->stats.kernel_launches++;
  CK(cudaGetLastError());
  return FSPT_OK;
}

int set_counts(Ctx* c, int band, int n_cont, int n_shadow) {  // also zeroes #hit, #miss and both cursors
  k_set_counts<<<1, 1, 0, band_stream(c, band)>>>(band_counts(c, band), n_cont, n_shadow, 0);
  CK(cudaGetLastError());
  return FSPT_OK;
}

// Adaptive sampling: the slots of the active pixels of rectangle f -> list, their number -> band_counts(band)[8], on the
// band's stream.  samples_per_pixel > 0: the wave's path count (S per active pixel) is set as set_counts does, and the
// samples are counted into d_stats[8].
int select_active(Ctx* c, int band, const FrameParams& f, int* list, int samples_per_pixel) {
  const cudaStream_t s = band_stream(c, band);
  int* counts = band_counts(c, band);
  const int P = f.rw * f.rh;
  CK(cudaMemsetAsync(counts + 8, 0, sizeof(int), s));
  k_select_active<<<(P + 255) / 256, 256, 0, s>>>(f, c->d_fb.p, c->d_m2.p, c->adapt_err, c->adapt_min, list, counts + 8,
                                                  samples_per_pixel ? c->d_stats.p + 8 : nullptr, samples_per_pixel);
  c->stats.kernel_launches++;
  CK(cudaGetLastError());
  if (samples_per_pixel) {
    k_set_counts<<<1, 1, 0, s>>>(counts, 0, 0, samples_per_pixel);
    CK(cudaGetLastError());
  }
  return FSPT_OK;
}

// The rectangle p renders and the slot -> pixel mapping that goes with it.
void set_rect(FrameParams& p, int rx0, int ry0, int rw, int rh) {
  p.rx0 = rx0; p.ry0 = ry0; p.rw = rw; p.rh = rh;
  p.tiled = (p.rw % 8 == 0 && p.rh % 4 == 0) ? 1 : 0;
  // slot -> pixel: one division by the tiles per row (dividend: a tile index) or by the row width (dividend: a pixel index)
  p.div_row = p.tiled ? make_fastdiv((unsigned)(p.rw >> 3), ((unsigned long long)p.rw * p.rh) >> 5)
                      : make_fastdiv((unsigned)p.rw, (unsigned long long)p.rw * p.rh);
}

FrameParams make_frame(const Ctx* c, const fspt_frame_params* f, bool whole_frame = false) {
  FrameParams p;
  for (int k = 0; k < 3; ++k) { p.eye[k] = f->eye[k]; p.dir[k] = f->dir[k]; }
  p.fov_scale = f->fov_scale; p.lens0 = f->lens_features[0]; p.lens1 = f->lens_features[1];
  p.env_theta = f->env_theta;
  {
    const v3 I = mk3(p.dir[0], p.dir[1], p.dir[2]);
    const v3 bx = normalize(cross(I, mk3(0.0f, 1.0f, 0.0f)));  // camera.fs:39
    const v3 by = normalize(cross(bx, I));                     // camera.fs:40
    p.basis_x[0] = bx.x; p.basis_x[1] = bx.y; p.basis_x[2] = bx.z;
    p.basis_y[0] = by.x; p.basis_y[1] = by.y; p.basis_y[2] = by.z;
  }
  p.width = c->width; p.height = c->height;
  if (whole_frame) set_rect(p, 0, 0, c->width, c->height);
  else set_rect(p, c->rx0, c->ry0, c->rw, c->rh);
  return p;
}

// Rand bases of one call -> device: [0,cap) camera, [cap,2cap) tracer.  The pinned staging is a ring; a slot is reused
// only after the DMA that read it has finished, so there is no stream synchronisation on the render path.
int stage_rand_bases(Ctx* c, const float* cam, const float* trace, int n) {
  if (n > c->rb_cap) {  // grow (rare): everything in flight must finish first
    CK(cudaStreamSynchronize(c->stream));
    c->rb_cap = std::max(n, 2 * c->rb_cap);
    CK(c->d_rb.fit(2 * (size_t)c->rb_cap * sizeof(float)));
    CK(c->h_rb.fit(Ctx::RB_SLOTS * 2 * (size_t)c->rb_cap * sizeof(float)));
  }
  if (n <= 0) return FSPT_OK;
  const int slot = c->rb_slot;
  c->rb_slot = (slot + 1) % Ctx::RB_SLOTS;
  CK(cudaEventSynchronize(c->ev_rb[slot]));  // returns at once unless RB_SLOTS calls are still queued
  float* h = c->h_rb.p + (size_t)slot * 2 * c->rb_cap;
  memcpy(h, cam, (size_t)n * sizeof(float));
  if (trace) memcpy(h + c->rb_cap, trace, (size_t)n * sizeof(float));
  CK(cudaMemcpyAsync(c->d_rb.p, h, 2 * (size_t)c->rb_cap * sizeof(float), cudaMemcpyHostToDevice, c->stream));
  CK(cudaEventRecord(c->ev_rb[slot], c->stream));
  return FSPT_OK;
}

// Paths a band must hold before a rectangle is split into two bands.  Measured on a B200: two bands of 0.32 M paths
// (800x800, 1 spp) render 3 % faster than one band, two of 29 M (1280x720, 64 spp) 0.6 % faster; smaller bands were
// not measured, so below 2^18 paths per band a wave stays one chain of launches.
#ifndef FSPT_BAND_MIN_PATHS
#define FSPT_BAND_MIN_PATHS (1 << 18)
#endif

// A wave of the rectangle fp is rendered as up to two row bands, each on its own stream (band_stream) with its own slice
// of the path arrays: every launch of a wave waits for the whole previous one, and the other band's CTAs fill the SMs
// while one band's launch ramps up or drains.  A pixel's samples do not depend on the rectangle that renders it, so
// the split changes no result.  The first band gets a multiple of 4 rows: a tiled rectangle gives two tiled bands.
int split_bands(const FrameParams& fp, int S, FrameParams band[2]) {
  const int rows0 = (fp.rh / 2) & ~3;
  band[0] = fp;
  if (rows0 == 0 || (size_t)S * fp.rw * rows0 < (size_t)FSPT_BAND_MIN_PATHS) return 1;
  band[1] = fp;
  set_rect(band[0], fp.rx0, fp.ry0, fp.rw, rows0);
  set_rect(band[1], fp.rx0, fp.ry0 + rows0, fp.rw, fp.rh - rows0);
  return 2;
}

// One wave.  Path records are dense arrays that ping-pong: set k = (array ps[k], counts band_counts()[2k .. 2k+1] =
// #records, #shadow rays); the shadow list holds record positions.  The bands' launches are enqueued interleaved, so
// that each stream always has its next launch queued behind the running one.
// Adaptive sampling: each band first lists its active pixels (k_select_active); the wave renders S samples of each,
// and its path count is known on the device only.  A wave with no active pixel still runs, with zero paths.
int render_wave(Ctx* c, const FrameParams& fp, uint32_t first_tick, int S, const float* rb_cam, const float* rb_trace) {
  FrameParams bfp[2];
  const int nb = split_bands(fp, S, bfp);
  BandSlice sl[2];
  int* list[2] = {nullptr, nullptr};
  int cur[2] = {0, 0};
  bool live[2] = {true, nb > 1};
  const bool adaptive = c->adapt_err > 0.0f;
  for (int b = 0, off = 0, px = 0; b < nb; ++b) {
    sl[b] = band_slice(c, (size_t)off);
    const int n_paths = S * bfp[b].rw * bfp[b].rh;
    off += n_paths;
    int rc;
    if (adaptive) {
      list[b] = c->d_list.p + px;
      px += bfp[b].rw * bfp[b].rh;
      rc = select_active(c, b, bfp[b], list[b], S);
    } else {
      rc = set_counts(c, b, n_paths, 0);
    }
    if (rc) return rc;
    // camera.fs + primary rays (tracer.fs:440), fused
    rc = launch_trace(c, b, sl[b], 0, true, false, &bfp[b], rb_cam, S, list[b]);
    if (rc) return rc;
  }
  int rc;
  ShadeArgs A;
  A.rb_trace = rb_trace;
  A.capped = c->d_stats.p + 3;
  A.n_samples = S;
  A.div_s = make_fastdiv((unsigned)S, c->wave_paths);
  A.max_refractions = c->max_refractions;
  A.anyhit = c->anyhit;
  const int hard_cap = FSPT_NUM_BOUNCES + 1 + (c->info.has_dielectric ? c->max_refractions + 2 : 0);
  // atlas of the last upload: an asynchronous upload's staging thread is joined HERE, with the primary traversal already
  // running on the GPU (the event it records has to exist before the stream can be made to wait on it); then the DMA
  // itself is waited for on the device (no-op once it has completed)
  // multi-GPU: the atlas travels to the other ranks now, behind the traversal.  (Phase 2 first: it joins the atlas thread
  // itself and, should the root's atlas part have failed, tells the other ranks instead of leaving them in the collective.)
  if ((rc = broadcast_phase2(c))) return rc;
  if ((rc = atlas_join(c))) return rc;
  A.sc = c->sc;  // (the atlas part sets the texture objects and table pointers)
  for (int b = 0; b < nb; ++b) CK(cudaStreamWaitEvent(band_stream(c, b), c->ev_atlas, 0));
  for (int it = 0; it < hard_cap && (live[0] || live[1]); ++it) {
    for (int b = 0; b < nb; ++b) {
      if (!live[b]) continue;
      const cudaStream_t s = band_stream(c, b);
      int* counts = band_counts(c, b);
      const int nxt = cur[b] ^ 1;
      CK(cudaMemsetAsync(counts + 2 * nxt, 0, 2 * sizeof(int), s));
      A.f = bfp[b];
      A.hit_flag = sl[b].hit_flag;
      A.shadow_rays_out = sl[b].shadow;
      A.sample_color = sl[b].sample_color;
      A.first = (it == 0);
      A.ps = sl[b].ps[cur[b]];
      A.ps_out = sl[b].ps[nxt];
      A.counts_in = counts + 2 * cur[b];
      A.counts_out = counts + 2 * nxt;
      A.tile_next = counts + 64;
      A.list = list[b];
      if ((rc = record_trace_begin(c, s, 1))) return rc;
      c->shade_kernels[c->sc.mat_tex != 0][adaptive]<<<c->shade_blocks, SHADE_THREADS, 1024, s>>>(A);
      record_trace_end(c, s);
      c->stats.kernel_launches++;
      CK(cudaGetLastError());
      cur[b] = nxt;
    }
    for (int b = 0; b < nb; ++b) {
      if (!live[b]) continue;
      const cudaStream_t s = band_stream(c, b);
      int* counts = band_counts(c, b);
      if (it >= FSPT_NUM_BOUNCES) {
        // every surviving path had i == NUM_BOUNCES: nothing was appended
        if (!c->info.has_dielectric) { live[b] = false; continue; }
        // Refractions do not count as bounces (`i--`, tracer.fs:488), so paths may survive.  The number of live paths
        // is copied out after every extra iteration, but the host reads the value of TWO iterations ago: the GPU always
        // has work queued and never waits for the host; at most two empty iterations (kernels that find zero items) are
        // wasted.  Each band polls and stops on its own.
        int* poll = c->h_poll.p + b * Ctx::POLL_SLOTS;
        const int k = it % Ctx::POLL_SLOTS;
        CK(cudaMemcpyAsync(poll + k, counts + 2 * cur[b], sizeof(int), cudaMemcpyDeviceToHost, s));
        CK(cudaEventRecord(c->ev_poll[b][k], s));
        if (it >= FSPT_NUM_BOUNCES + 2) {
          const int k2 = (it - 2) % Ctx::POLL_SLOTS;
          CK(cudaEventSynchronize(c->ev_poll[b][k2]));
          if (poll[k2] == 0) { live[b] = false; continue; }
        }
      }
      CK(cudaMemsetAsync(counts + 32, 0, sizeof(int), s));  // fetch cursor
      rc = launch_trace(c, b, sl[b], cur[b], true, false);  // tracer.fs:501,507
      if (rc) return rc;
    }
  }
  for (int b = 0; b < nb; ++b) {
    const FrameParams& f = bfp[b];
    const int P = f.rw * f.rh;
    if (adaptive)
      k_accumulate_active<<<(P + 255) / 256, 256, 0, band_stream(c, b)>>>(f, list[b], band_counts(c, b) + 8,
                                                                          sl[b].sample_color, c->d_fb.p,
                                                                          c->d_last_color.p, c->d_m2.p, S, c->sanitize);
    else
      k_accumulate<<<(P + 255) / 256, 256, 0, band_stream(c, b)>>>(sl[b].sample_color, c->d_fb.p, c->d_last_color.p,
                                                                   f.rx0, f.ry0, f.rw, f.rh, f.width, S, first_tick,
                                                                   c->accum_mode, c->sanitize);
    c->stats.kernel_launches++;
    CK(cudaGetLastError());
  }
  return FSPT_OK;
}

// ---- NCCL, resolved at run time ----------------------------------------------------------------------------------
// The library has no link-time dependency on NCCL: a single-GPU host never loads it.  dlopen("libnccl.so.2") returns
// the copy already mapped into the process when there is one (e.g. the one a PyTorch host brought along), else the
// system library.
struct NcclApi {
  void* handle = nullptr;
  ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
  ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  ncclResult_t (*Reduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*Broadcast)(const void*, void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*GroupStart)() = nullptr;
  ncclResult_t (*GroupEnd)() = nullptr;
  const char* (*GetErrorString)(ncclResult_t) = nullptr;
  std::string error;
};
NcclApi* nccl_api() {
  static NcclApi api;
  static std::once_flag once;
  std::call_once(once, []() {
    const char* names[] = {getenv("FSPT_NCCL_LIB"), "libnccl.so.2", "libnccl.so"};
    for (const char* n : names) {
      if (!n || !*n) continue;
      api.handle = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
      if (api.handle) break;
    }
    if (!api.handle) { api.error = std::string("dlopen(libnccl.so.2) failed: ") + dlerror(); return; }
    auto sym = [&](const char* name) {
      void* p = dlsym(api.handle, name);
      if (!p && api.error.empty()) api.error = std::string("NCCL symbol missing: ") + name;
      return p;
    };
    api.GetUniqueId = reinterpret_cast<decltype(api.GetUniqueId)>(sym("ncclGetUniqueId"));
    api.CommInitRank = reinterpret_cast<decltype(api.CommInitRank)>(sym("ncclCommInitRank"));
    api.CommDestroy = reinterpret_cast<decltype(api.CommDestroy)>(sym("ncclCommDestroy"));
    api.Reduce = reinterpret_cast<decltype(api.Reduce)>(sym("ncclReduce"));
    api.Broadcast = reinterpret_cast<decltype(api.Broadcast)>(sym("ncclBroadcast"));
    api.GroupStart = reinterpret_cast<decltype(api.GroupStart)>(sym("ncclGroupStart"));
    api.GroupEnd = reinterpret_cast<decltype(api.GroupEnd)>(sym("ncclGroupEnd"));
    api.GetErrorString = reinterpret_cast<decltype(api.GetErrorString)>(sym("ncclGetErrorString"));
  });
  return &api;
}
#define NK(call)                                                                                               \
  do {                                                                                                         \
    ncclResult_t r_ = (call);                                                                                  \
    if (r_ != ncclSuccess) return fail(c, FSPT_E_NCCL, "%s failed: %s", #call, nccl_api()->GetErrorString(r_)); \
  } while (0)

void comm_free(Ctx* c) {
  if (c->comm) nccl_api()->CommDestroy(c->comm);
  c->comm = nullptr;
  c->comm_rank = 0; c->comm_world = 1;
}

// what a receiving rank has to know before the buffers of fspt_scene_broadcast arrive
struct SceneHeader {
  SceneInfo scene;
  int32_t magic;
};

// what a receiving rank has to know before the atlas part of fspt_scene_broadcast arrives (phase 2)
struct SceneHeader2 {
  AtlasInfo atlas;
  int32_t magic;
};

// The scene resident on `root` -> every other rank, device to device over NVLink: the records fspt_scene_upload built
// (Node64, Tri48, ShadeRec, bins, layer / material tables) and linear copies of the environment and atlas arrays.  One
// host stages and uploads a scene once instead of every rank repeating the same 200 MB of host work.
//
// Two phases, like the upload itself.  Phase 1 (here, on the context's stream): what the traversal kernel needs -- and
// the environment.  Phase 2 (the atlas and its tables, on the copy stream) is DEFERRED to the point where the root's
// atlas is needed anyway: the first shading launch of the next fspt_render, behind its primary traversal launch (or the
// next fspt_synchronize / fspt_reduce_accum / upload / broadcast, whichever comes first -- every rank reaches one of them,
// in the same order relative to the other collectives).  An asynchronous upload on the root therefore overlaps its atlas
// transfer with the primary traversal on EVERY rank, and the root's host is not held in the broadcast call.
int broadcast_phase2(Ctx* c) {
  if (c->bcast_pending_root < 0) return FSPT_OK;
  const int root = c->bcast_pending_root;
  c->bcast_pending_root = -1;
  const bool is_root = c->comm_rank == root;
  NcclApi* N = nccl_api();
  SceneHeader2 h;
  memset(&h, 0, sizeof h);
  static_assert(sizeof(SceneHeader2) <= 128, "header buffer");
  uint8_t* d_hdr2 = c->d_hdr.p + 256;
  // the collectives of one communicator run one after the other: this one starts behind phase 1 (its last collective
  // recorded the event), not behind the traversal launch that may have been enqueued since
  CK(cudaStreamWaitEvent(c->copy_stream, c->ev_bcast, 0));
  if (is_root) {
    int rcj = atlas_join(c);  // the root's atlas part ends here at the latest; its outcome travels in the header
    if (rcj) h.magic = -1;    // the ranks must not wait for an atlas that will not come
    else {
      h.atlas = c->atlas_info;
      h.magic = 0x46535032;
    }
    CK(cudaMemcpyAsync(d_hdr2, &h, sizeof h, cudaMemcpyHostToDevice, c->copy_stream));
    NK(N->Broadcast(d_hdr2, d_hdr2, sizeof h, ncclUint8, root, c->comm, c->copy_stream));
    if (rcj) return rcj;
  } else {
    NK(N->Broadcast(d_hdr2, d_hdr2, sizeof h, ncclUint8, root, c->comm, c->copy_stream));
    CK(cudaMemcpyAsync(&h, d_hdr2, sizeof h, cudaMemcpyDeviceToHost, c->copy_stream));
    CK(cudaStreamSynchronize(c->copy_stream));
    if (h.magic != 0x46535032) { c->has_scene = false; return fail(c, FSPT_E_NCCL, "fspt_scene_broadcast: rank %d has no atlas to send (its upload failed)", root); }
  }
  const AtlasInfo& a = h.atlas;
  const size_t texel = a.interleaved ? 16 : 4;
  const size_t atlas_bytes = (size_t)a.res * a.res * texel * (size_t)a.layers;
  CK(c->d_lin.fit(atlas_bytes));
  uint8_t* lin = c->d_lin.p;
  cudaMemcpy3DParms cp = {};
  cp.extent = make_cudaExtent(a.res, a.res, a.layers);
  cp.kind = cudaMemcpyDeviceToDevice;
  if (is_root) {
    // the atlas DMA of the upload runs on this same stream (in order)
    cp.srcArray = (a.interleaved ? c->mat : c->atlas).arr;
    cp.dstPtr = make_cudaPitchedPtr(lin, (size_t)a.res * texel, a.res, a.res);
    CK(cudaMemcpy3DAsync(&cp, c->copy_stream));
  } else {
    // storage on the receiving side: same reuse rules as fspt_scene_upload
    c->has_scene = false;
    CK(c->d_layer_info.fit(a.bytes_layer_info));
    CK(c->d_mat_info.fit(a.bytes_mat_info));
    CK(fit_atlas(c, a.interleaved, a.res, a.layers, false));
  }
  NK(N->GroupStart());
  NK(N->Broadcast(c->d_layer_info.p, c->d_layer_info.p, a.bytes_layer_info, ncclUint8, root, c->comm, c->copy_stream));
  NK(N->Broadcast(c->d_mat_info.p, c->d_mat_info.p, a.bytes_mat_info, ncclUint8, root, c->comm, c->copy_stream));
  NK(N->Broadcast(lin, lin, atlas_bytes, ncclUint8, root, c->comm, c->copy_stream));
  NK(N->GroupEnd());
  c->stats.kernel_launches += 4;
  if (!is_root) {
    cp.srcPtr = make_cudaPitchedPtr(lin, (size_t)a.res * texel, a.res, a.res);
    cp.dstArray = (a.interleaved ? c->mat : c->atlas).arr;
    CK(cudaMemcpy3DAsync(&cp, c->copy_stream));
    publish_atlas(c, a);
    c->has_scene = true;
  }
  // what the first shading launch waits for; later collectives on the context's stream come behind it as well
  CK(cudaEventRecord(c->ev_atlas, c->copy_stream));
  CK(cudaStreamWaitEvent(c->stream, c->ev_atlas, 0));
  return FSPT_OK;
}

int pull_stats(Ctx* c) {
  unsigned long long h[9];
  CK(cudaMemcpy(h, c->d_stats.p, sizeof h, cudaMemcpyDeviceToHost));
  c->stats.rays = h[0]; c->stats.node_visits = h[1]; c->stats.leaf_visits = h[2]; c->stats.capped_paths = h[3];
  c->adaptive_samples = h[8];
  c->stats.last_rays = h[0] - h[4]; c->stats.last_node_visits = h[1] - h[5]; c->stats.last_leaf_visits = h[2] - h[6];
  return FSPT_OK;
}

}  // namespace

extern "C" {

int fspt_abi_version(void) { return FSPT_ABI_VERSION; }

const char* fspt_last_error(const fspt_ctx* ctx) {
  if (!ctx) return g_create_error.c_str();
  return reinterpret_cast<const Ctx*>(ctx)->error.c_str();
}

int fspt_create(fspt_ctx** out, int32_t width, int32_t height, int32_t device) {
  Ctx* c = nullptr;
  if (!out || width <= 0 || height <= 0 || (int64_t)width * height > (1 << 27))
    return fail(c, FSPT_E_INVALID, "fspt_create: bad arguments (%d x %d)", width, height);
  if (int rc = fspt_device_check(device)) return rc;
  c = new Ctx();
  c->device = device;
  c->width = width; c->height = height; c->n_pixels = width * height;
  c->rx0 = c->ry0 = 0; c->rw = width; c->rh = height;
  auto init = [c]() -> int {
    const size_t px16 = (size_t)c->n_pixels * 16;
    CK(cudaSetDevice(c->device));
    CK(cudaDeviceGetAttribute(&c->sm_count, cudaDevAttrMultiProcessorCount, c->device));
    for (Stream* s : {&c->stream, &c->copy_stream, &c->stream2}) CK(s->create(cudaStreamNonBlocking));
    for (Event* e : {&c->ev_fork, &c->ev_join, &c->ev_atlas, &c->ev_env, &c->ev_bcast}) CK(e->create(cudaEventDisableTiming));
    for (Event* e : {&c->ev_begin, &c->ev_end, &c->ev_red0, &c->ev_red1}) CK(e->create(cudaEventDefault));
    CK(c->d_fb.fit(px16));
    CK(cudaMemset(c->d_fb.p, 0, px16));
    CK(c->d_last_color.fit(px16));
    CK(c->d_cam_pos.fit(px16));
    CK(c->d_cam_dir.fit(px16));
    CK(c->d_rgba8.fit((size_t)c->n_pixels * 4));
    return alloc_wave(c);
  };
  if (int rc = init()) { g_create_error = c->error; fspt_destroy(reinterpret_cast<fspt_ctx*>(c)); return rc; }
  // persistent grids: resident CTAs per SM x SM count.  The traversal kernel keeps its short stacks and a few per-ray
  // values in shared memory; everything else of the unified array should stay L1 (BVH nodes and leaf blocks live
  // there), so the carveout is set to what the resident CTAs need and no more.
  int max_smem_sm = 0;
  cudaDeviceGetAttribute(&max_smem_sm, cudaDevAttrMaxSharedMemoryPerMultiprocessor, device);
  auto persistent = [&](auto kernel) {
    int per_sm = 0;
    cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, TRACE_THREADS, 0);
    per_sm = std::max(1, per_sm);
    cudaFuncAttributes fa{};
    cudaFuncGetAttributes(&fa, kernel);
    if (max_smem_sm > 0) {
      const size_t need = (size_t)per_sm * (fa.sharedSizeBytes + 1024);  // + the per-CTA reservation
      const int pct = (int)std::min<size_t>(100, (need * 100 + (size_t)max_smem_sm - 1) / (size_t)max_smem_sm);
      cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, pct);
    }
    return per_sm * c->sm_count;
  };
  for (auto& row : c->trace_kernels)
    for (TraceKernel& k : row) k.blocks = persistent(k.fn);
  int per_sm = 0;
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_shade<true>, SHADE_THREADS, 1024);
  c->shade_blocks = std::max(1, per_sm) * c->sm_count;
  *out = reinterpret_cast<fspt_ctx*>(c);
  return FSPT_OK;
}

void fspt_destroy(fspt_ctx* ctx) {
  Ctx* c = reinterpret_cast<Ctx*>(ctx);
  if (!c) return;
  cudaSetDevice(c->device);
  if (c->atlas_thread.joinable()) c->atlas_thread.join();
  c->bcast_pending_root = -1;  // (no collective in a destructor)
  for (const Stream* s : {&c->stream, &c->copy_stream, &c->stream2})
    if (*s) cudaStreamSynchronize(*s);
  comm_free(c);
  delete c;  // frees the host workers, texture objects, buffers, arrays, events and streams (Ctx's member order)
}

// fspt_scene_upload / fspt_scene_upload_async.
// Order of work (round 2, second half: the geometry used to be staged next to the atlas by a quarter of the host
// threads and DMA'd only when all of it was ready, which put ~3 ms between the call and the first traversal launch):
//   1. pre-passes over nodes and triangles (parallel): interior-record numbering, material ids;
//   2. geometry records (Node64 / Tri48 / ShadeRec), bins and environment: built chunk by chunk by ALL host workers into
//      a ring of pinned slots, every chunk DMA'd the moment it is complete -- the traversal kernel's inputs are on
//      their way before anything else is touched, and a 10 M-triangle scene (2.6 GB of records) streams through
//      256 MB of pinned memory instead of a pageable copy;
//   3. the atlas part (stage_atlas): inline, or -- async_atlas -- on the context's atlas thread after this function has
//      returned; every other buffer of the scene has been consumed by then.
static int scene_upload_impl(fspt_ctx* ctx, const fspt_scene_desc* s, bool async_atlas) {
  Ctx* c = reinterpret_cast<Ctx*>(ctx);
  const bool timing = getenv("FSPT_TIMING") != nullptr;
  auto t_prev = std::chrono::steady_clock::now();
  auto lap = [&](const char* what) {
    if (!timing) return;
    auto now = std::chrono::steady_clock::now();
    fprintf(stderr, "[fspt upload] %-28s %7.2f ms\n", what, std::chrono::duration<double, std::milli>(now - t_prev).count());
    t_prev = now;
  };
  if (!c) return FSPT_E_INVALID;
  if (!s || !s->bvh || !s->triangles || !s->materials || !s->normals || !s->uvs || !s->atlas || !s->env || !s->radiance_bins)
    return fail(c, FSPT_E_INVALID, "scene_upload: NULL buffer");
  if (s->n_nodes <= 0 || s->n_triangles <= 0 || s->atlas_res <= 0 || s->atlas_layers <= 0 || s->env_width <= 0 ||
      s->env_height <= 0 || s->env_bins <= 0)
    return fail(c, FSPT_E_INVALID, "scene_upload: non-positive size (an environment with >= 1 bin is mandatory, main.js:303-308)");
  if (s->leaf_size != 4) return fail(c, FSPT_E_INVALID, "scene_upload: LEAF_SIZE must be 4 (main.js:45), got %d", s->leaf_size);
  CK(cudaSetDevice(c->device));
  if (int rcb = broadcast_phase2(c)) return rcb;  // (a broadcast nobody rendered from: finish it before its source goes away)
  (void)atlas_join(c);  // the atlas thread of the previous upload still reads the pinned blocks and the arrays
  CK(cudaStreamSynchronize(c->stream));
  CK(cudaStreamSynchronize(c->copy_stream));
  c->has_scene = false;  // device buffers, arrays and texture objects of the previous scene are reused when they fit
  lap("sync");
  const int N = s->n_nodes, T = s->n_triangles;
  const int L = s->atlas_layers;
  // host threads for staging: all cores of a single-process host; one process per GPU shares them
  // (dist.share_host_threads sets FSPT_UPLOAD_THREADS = cores / processes on this node)
  int hw = (int)std::max(4u, std::min(32u, std::thread::hardware_concurrency()));
  if (const char* e = getenv("FSPT_UPLOAD_THREADS")) hw = std::max(4, std::min(64, atoi(e)));
  if (!c->pool) { const int device = c->device; c->pool = std::make_unique<HostPool>([device]() { cudaSetDevice(device); }); }
  HostPool& pool = *c->pool;
  // ---- pre-passes (scene_pack.h): interior-record numbering, material ids, depth / tree check
  ScenePrepass pre;
  {
    const int rcp = scene_prepass(pool, hw, s, pre);
    if (rcp) return fail(c, rcp, "%s", pre.error.c_str());
  }
  std::vector<std::array<int, 4>>& mats = pre.mats;
  const size_t NI = pre.NI();
  lap("node + material pre-pass");

  // ---- pinned block for the small tables and the environment (kept between uploads)
  auto al = [](size_t x) { return (x + 255) & ~(size_t)255; };
  const size_t env_bytes = (size_t)s->env_width * s->env_height * 4;
  const size_t o_bins = 0, o_layer = o_bins + al((size_t)s->env_bins * 16), o_mat = o_layer + al((size_t)L * 8),
               o_matsrc = o_mat + al(std::max<size_t>(32, mats.size() * 32)),
               o_env = o_matsrc + al(std::max<size_t>(32, mats.size() * sizeof(MatSrc))), small_bytes = o_env + al(env_bytes);
  CK(c->h_geo.fit(small_bytes));
  uint8_t* hg = c->h_geo.p;
  float* bins = reinterpret_cast<float*>(hg + o_bins);
  const size_t n_mat_info = std::max<size_t>(8, mats.size() * 8);
  // ---- device buffers, environment array
  SceneInfo si;
  si.bytes_nodes = std::max<size_t>(NI, 1) * 64;
  si.bytes_tris = (size_t)(T + 3) * 48;
  si.bytes_shade = (size_t)T * 192;
  si.bytes_bins = (size_t)s->env_bins * 16;
  si.scene_bytes = (size_t)N * 36 + (size_t)T * (36 + 48 + 108 + 24) + (size_t)s->atlas_res * s->atlas_res * 4 * L +
                   env_bytes + (size_t)s->env_bins * 8;
  si.root_ref = pre.ref[0];
  si.n_tris = T; si.n_interior = (int)NI;
  si.atlas_res = s->atlas_res; si.atlas_layers = L; si.env_w = s->env_width; si.env_h = s->env_height;
  si.n_bins = s->env_bins;
  si.has_dielectric = pre.dielectric;
  int rc_;
  if ((rc_ = fit_scene(c, si))) return rc_;
  // ---- work items of the staging region: bands of the environment (+ the bins), node chunks, triangle chunks -- each
  // DMA'd the moment it is complete -- and, behind them, the constant-layer scan of the atlas, which the workers that
  // run out of geometry pick up.  Chunks are sized so that a small scene still gives every worker a few items; each
  // geometry chunk owns one slot of the pinned ring.
  const int workers = hw;
  const int tri_chunk = (int)std::max<size_t>(1024, std::min<size_t>(16384, ((size_t)T + 3) / (4 * (size_t)workers) + 1));
  const int node_chunk = (int)std::max<size_t>(4096, std::min<size_t>(65536, NI / (4 * (size_t)workers) + 1));
  const int n_node_items = NI ? (int)((NI + node_chunk - 1) / node_chunk) : 1;
  const int n_tri_items = (T + 3 + tri_chunk - 1) / tri_chunk;
  const int n_env_items = std::max(1, std::min(s->env_height, (int)(env_bytes >> 20)));  // ~1 MB of rows each
  const int n_geo_items = n_node_items + n_tri_items;
  // (a page-locked atlas under an asynchronous upload: the scan is all the host work the atlas part has left, and it
  // should not hold up this function's return -- it moves to the atlas thread)
  const bool atlas_pinned = host_is_pinned(s->atlas);
  const bool scan_here = !(async_atlas && atlas_pinned);
  const int n_scan_items = scan_here ? L * SCAN_BANDS : 0;
  const int n_items = n_env_items + n_geo_items + n_scan_items;
  const size_t layer_texels = (size_t)s->atlas_res * s->atlas_res;
  std::vector<std::atomic<int>> varied((size_t)L);
  for (auto& v : varied) v.store(0);
  const size_t slot_bytes = al(std::max<size_t>((size_t)node_chunk * 64, (size_t)tri_chunk * (48 + 192)));
  int n_slots = (int)std::max<size_t>(1, std::min<size_t>((size_t)n_geo_items, std::max<size_t>(2 * (size_t)workers, ((size_t)256 << 20) / slot_bytes)));
  if (const char* e = getenv("FSPT_RING_SLOTS")) n_slots = std::max(1, std::min(n_slots, atoi(e)));  // test knob: force slot reuse
  const bool ring_wraps = n_geo_items > n_slots;  // otherwise every chunk has a slot of its own and no event is needed
  CK(c->h_ring.fit(slot_bytes * (size_t)n_slots));
  while ((int)c->ev_ring.size() < n_slots) {
    Event e;
    CK(e.create(cudaEventDisableTiming));
    c->ev_ring.push_back(std::move(e));
  }
  lap("buffers + pinned ring");
  struct GeoStatus { int code = FSPT_OK; char msg[192] = {0}; } geo;
  std::mutex geo_mu;
  auto geo_fail = [&](int code, const char* fmt, int a0, int a1, int a2) {
    std::lock_guard<std::mutex> g(geo_mu);
    if (geo.code == FSPT_OK) { geo.code = code; snprintf(geo.msg, sizeof geo.msg, fmt, a0, a1, a2); }
  };
  std::atomic<int> dma_err(0);
  // (No lock around the enqueues: the runtime is thread-safe, and a slot's event only has to follow the slot's own copies,
  // which the recording thread enqueued itself.  A mutex held across the two or three calls of an item serialised ~60
  // items x ~12 us on the bench scene -- most of the region's 1.4 ms.)
  const bool src_env_pinned = host_is_pinned(s->env);
  std::vector<std::atomic<int>> slot_done((size_t)n_slots);  // last item whose copies have been enqueued from the slot
  for (auto& v : slot_done) v.store(-1);
  pool.run(n_items, workers, [&](int item) {
    if (item < n_env_items) {  // a band of environment rows (+ the bins): their own pinned block
      if (item == 0)
        for (size_t i = 0; i < (size_t)s->env_bins * 4; ++i) bins[i] = (float)s->radiance_bins[i];  // vec4(radianceBins[idx]), tracer.fs:424
      const size_t pitch = (size_t)s->env_width * 4;
      const int y0 = (int)((long long)s->env_height * item / n_env_items), y1 = (int)((long long)s->env_height * (item + 1) / n_env_items);
      const uint8_t* src = s->env + y0 * pitch;   // page-locked by the caller (fspt_host_register): DMA'd where it lies
      if (!src_env_pinned) { memcpy(hg + o_env + y0 * pitch, src, (size_t)(y1 - y0) * pitch); src = hg + o_env + y0 * pitch; }
      cudaError_t e = item == 0 ? cudaMemcpyAsync(c->d_bins.p, bins, si.bytes_bins, cudaMemcpyHostToDevice, c->stream) : cudaSuccess;
      if (e == cudaSuccess)
        e = cudaMemcpy2DToArrayAsync(c->env.arr, 0, y0, src, pitch, pitch, y1 - y0, cudaMemcpyHostToDevice, c->stream);
      if (e != cudaSuccess) dma_err.store((int)e);
      return;
    }
    if (item >= n_env_items + n_geo_items) {  // atlas: constant-layer scan
      scan_layer_band(s->atlas, layer_texels, item - n_env_items - n_geo_items, varied.data());
      return;
    }
    // ring slot of this chunk: free once the copies of the chunk that used it last have completed
    const int ring_item = item - n_env_items, slot = ring_item % n_slots;
    if (ring_item >= n_slots) {
      while (slot_done[slot].load(std::memory_order_acquire) != ring_item - n_slots) std::this_thread::yield();
      cudaEventSynchronize(c->ev_ring[slot]);
    }
    uint8_t* hs = c->h_ring.p + (size_t)slot * slot_bytes;
    cudaError_t e = cudaSuccess;
    if (ring_item < n_node_items) {
      const size_t k0 = (size_t)ring_item * node_chunk, k1 = std::min(NI, k0 + node_chunk);
      float* nodes = reinterpret_cast<float*>(hs);
      int bl = 0, br = 0;
      const int bad = pack_node_chunk(s, pre, k0, k1, nodes, &bl, &br);
      if (bad >= 0) geo_fail(FSPT_E_INVALID, "node %d: child index out of range (%d, %d)", bad, bl, br);
      const size_t bytes = NI ? (k1 - k0) * 64 : 64;
      e = cudaMemcpyAsync(c->d_nodes.p + k0 * 64, nodes, bytes, cudaMemcpyHostToDevice, c->stream);
      if (e == cudaSuccess && ring_wraps) e = cudaEventRecord(c->ev_ring[slot], c->stream);
    } else {
      const int t0 = (ring_item - n_node_items) * tri_chunk, t1 = std::min(T + 3, t0 + tri_chunk), ts = std::min(T, t1);
      float* tris = reinterpret_cast<float*>(hs);
      float* shade = reinterpret_cast<float*>(hs + (size_t)tri_chunk * 48);
      pack_tri_chunk(s, pre, t0, t1, tris, shade);
      e = cudaMemcpyAsync(c->d_tris.p + (size_t)t0 * 48, tris, (size_t)(t1 - t0) * 48, cudaMemcpyHostToDevice, c->stream);
      if (e == cudaSuccess && ts > t0)
        e = cudaMemcpyAsync(c->d_shade.p + (size_t)t0 * 192, shade, (size_t)(ts - t0) * 192, cudaMemcpyHostToDevice, c->stream);
      if (e == cudaSuccess && ring_wraps) e = cudaEventRecord(c->ev_ring[slot], c->stream);
    }
    if (e != cudaSuccess) dma_err.store((int)e);
    slot_done[slot].store(ring_item, std::memory_order_release);
  });
  if (dma_err.load()) return fail(c, FSPT_E_CUDA, "geometry upload failed: %s", cudaGetErrorString((cudaError_t)dma_err.load()));
  c->env_in_place = src_env_pinned;
  if (src_env_pinned) CK(cudaEventRecord(c->ev_env, c->stream));
  lap("geometry + env + layer scan");
  if ((rc_ = publish_scene(c, si))) return rc_;
  // ---- the atlas part: here, or on the context's atlas thread (the caller's atlas stays borrowed until it is joined).
  // Measured alternatives (e2e step of the bench scene, asynchronous upload, 29.4 ms as built): the layer scan inside the
  // atlas part instead of the staging region 29.8 (the upload returns 0.2 ms earlier but the atlas lands 0.7 ms later, and
  // the first shading launch waits for that); the whole atlas part started before the geometry staging on workers of
  // its own 32.5 (32 threads on 16 cores: the geometry, which the first traversal launch waits for, takes 3 ms).
  AtlasJob job;
  job.atlas = s->atlas; job.L = L; job.R = s->atlas_res;
  job.mats = std::move(mats);
  job.layer_info = reinterpret_cast<uint32_t*>(hg + o_layer);
  job.mat_info = reinterpret_cast<int32_t*>(hg + o_mat);
  job.n_mat_info = n_mat_info;
  job.mat_src = reinterpret_cast<MatSrc*>(hg + o_matsrc);
  if (scan_here) {
    job.varied.resize((size_t)L);
    for (int l = 0; l < L; ++l) job.varied[l] = (uint8_t)varied[l].load();
  }
  job.src_pinned = atlas_pinned;
  job.workers = hw;
  job.timing = timing;
  c->atlas_rc = FSPT_OK;
  c->atlas_in_place = false;
  struct StagingGuard {  // an error return below must not leave the atlas thread reading the caller's buffer
    Ctx* c; bool ok = false;
    ~StagingGuard() { if (!ok && c->atlas_thread.joinable()) c->atlas_thread.join(); }
  } staging_guard{c};
  if (async_atlas) {
    const int device = c->device;
    c->atlas_thread = std::thread([c, device, job = std::move(job)]() {
      cudaSetDevice(device);
      c->atlas_rc = stage_atlas(c, job);
    });
    lap("atlas part handed to its thread");
  } else {
    if ((rc_ = stage_atlas(c, job))) { c->error = "atlas upload: " + c->atlas_error; return rc_; }
    lap("atlas part");
  }
  if (geo.code != FSPT_OK) return fail(c, geo.code, "%s", geo.msg);
  // no synchronisation: everything the DMA engines still read lives in the context's pinned blocks, which the next
  // upload (and destroy) only touch after synchronising the streams; work enqueued by fspt_render waits in order
  if (timing && !async_atlas) { CK(cudaStreamSynchronize(c->stream)); CK(cudaStreamSynchronize(c->copy_stream)); lap("sync (timing only)"); }
  c->has_scene = true;
  staging_guard.ok = true;
  if (!async_atlas) {  // a synchronous upload has consumed every buffer when it returns, page-locked ones included
    int rcw = release_borrowed(c);
    if (rcw) return rcw;
  }
  return FSPT_OK;
}

int fspt_scene_upload(fspt_ctx* ctx, const fspt_scene_desc* s) { return scene_upload_impl(ctx, s, false); }
int fspt_scene_upload_async(fspt_ctx* ctx, const fspt_scene_desc* s) { return scene_upload_impl(ctx, s, true); }
int fspt_debug_pack_scene(const fspt_scene_desc* s, float* node64_out, float* tri48_out, float* shaderec_out,
                          int32_t* mat_id_out, int32_t* info_out, int32_t n_threads) {
  if (!s || !s->bvh || !s->triangles || !s->materials || !s->normals || !s->uvs || !info_out || s->n_nodes <= 0 ||
      s->n_triangles <= 0 || s->atlas_layers <= 0)
    return FSPT_E_INVALID;
  const int hw = std::max(1, std::min(64, n_threads > 0 ? n_threads : (int)std::thread::hardware_concurrency()));
  HostPool pool;
  ScenePrepass pre;
  const int rc = scene_prepass(pool, hw, s, pre);
  if (rc) { g_create_error = pre.error; return rc; }
  const size_t NI = pre.NI();
  info_out[0] = (int32_t)NI; info_out[1] = (int32_t)pre.mats.size(); info_out[2] = pre.ref[0];
  info_out[3] = pre.dielectric ? 1 : 0; info_out[4] = pre.max_depth;
  if (!node64_out) return FSPT_OK;  // first call: sizes only
  if (!tri48_out || !shaderec_out) return FSPT_E_INVALID;
  const int T = s->n_triangles;
  const size_t node_chunk = 4096;
  const int tri_chunk = 1024;
  const int n_node_items = NI ? (int)((NI + node_chunk - 1) / node_chunk) : 1, n_tri_items = (T + 3 + tri_chunk - 1) / tri_chunk;
  std::atomic<int> bad(-1);
  pool.run(n_node_items + n_tri_items, hw, [&](int item) {
    if (item < n_node_items) {
      const size_t k0 = (size_t)item * node_chunk, k1 = std::min(NI, k0 + node_chunk);
      int bl = 0, br = 0;
      const int b = pack_node_chunk(s, pre, k0, k1, node64_out + k0 * 16, &bl, &br);
      if (b >= 0) { int exp = -1; bad.compare_exchange_strong(exp, b); }
      return;
    }
    const int t0 = (item - n_node_items) * tri_chunk, t1 = std::min(T + 3, t0 + tri_chunk);
    pack_tri_chunk(s, pre, t0, t1, tri48_out + (size_t)t0 * 12, shaderec_out + (size_t)t0 * 48);
  });
  if (bad.load() >= 0) { g_create_error = "node " + std::to_string(bad.load()) + ": child index out of range"; return FSPT_E_INVALID; }
  if (mat_id_out) memcpy(mat_id_out, pre.mat_id.data(), (size_t)T * 4);
  return FSPT_OK;
}

int fspt_host_register(void* p, uint64_t bytes) {
  if (!p || !bytes) return FSPT_E_INVALID;
  cudaError_t e = cudaHostRegister(p, bytes, cudaHostRegisterPortable);
  if (e == cudaErrorHostMemoryAlreadyRegistered) { (void)cudaGetLastError(); return FSPT_OK; }
  if (e != cudaSuccess) { (void)cudaGetLastError(); g_create_error = std::string("cudaHostRegister: ") + cudaGetErrorString(e); return FSPT_E_CUDA; }
  return FSPT_OK;
}
int fspt_host_unregister(void* p) {
  if (!p) return FSPT_E_INVALID;
  cudaError_t e = cudaHostUnregister(p);
  if (e != cudaSuccess) { (void)cudaGetLastError(); g_create_error = std::string("cudaHostUnregister: ") + cudaGetErrorString(e); return FSPT_E_CUDA; }
  return FSPT_OK;
}

int fspt_scene_upload_wait(fspt_ctx* ctx) {
  Ctx* c = reinterpret_cast<Ctx*>(ctx);
  if (!c) return FSPT_E_INVALID;
  CK(cudaSetDevice(c->device));
  if (int rc = atlas_join(c)) return rc;
  return release_borrowed(c);
}

int fspt_clear(fspt_ctx* ctx) {
  Ctx* c = reinterpret_cast<Ctx*>(ctx);
  if (!c) return FSPT_E_INVALID;
  CK(cudaSetDevice(c->device));
  CK(cudaMemsetAsync(c->d_fb.p, 0, (size_t)c->n_pixels * 16, c->stream));
  if (c->d_m2.p) {  // adaptive sampling has been on: its moment and sample count start again too
    CK(cudaMemsetAsync(c->d_m2.p, 0, (size_t)c->n_pixels * sizeof(float), c->stream));
    CK(cudaMemsetAsync(c->d_stats.p + 8, 0, sizeof(unsigned long long), c->stream));
    c->adaptive_samples = 0;
  }
  c->next_tick = 0;
  c->accum_samples = 0;
  c->stats.samples = 0;
  return FSPT_OK;
}

int fspt_render(fspt_ctx* ctx, const fspt_frame_params* frame, uint32_t first_tick, int32_t n_samples,
                const float* rand_base_camera, const float* rand_base_tracer) {
  Ctx* c = reinterpret_cast<Ctx*>(ctx);
  if (!c) return FSPT_E_INVALID;
  if (!frame || n_samples < 0 || (n_samples > 0 && (!rand_base_camera || !rand_base_tracer)))
    return fail(c, FSPT_E_INVALID, "fspt_render: bad arguments");
  if (!c->has_scene) return fail(c, FSPT_E_STATE, "fspt_render before fspt_scene_upload");
  const bool adaptive = c->adapt_err > 0.0f;
  if (adaptive && c->accum_mode != 1)
    return fail(c, FSPT_E_STATE, "fspt_render: adaptive sampling needs the sum accumulation mode (fspt_set_accum_mode(ctx, 1))");
  CK(cudaSetDevice(c->device));
  const FrameParams fp = make_frame(c, frame);
  c->ev_trace_used = 0;
  CK(cudaMemcpyAsync(c->d_stats.p + 4, c->d_stats.p, 4 * sizeof(unsigned long long), cudaMemcpyDeviceToDevice, c->stream));
  // all rand bases of this call go up in one copy: [0,cap) camera, [cap,2cap) tracer
  {
    int rc0 = stage_rand_bases(c, rand_base_camera, rand_base_tracer, n_samples);
    if (rc0) return rc0;
  }
  CK(cudaEventRecord(c->ev_begin, c->stream));
  // the second band's stream starts behind the rand-base copy and is joined back before ev_end, so everything after the
  // render (timing, reduce, post-pass, read-back, collectives) stays ordered on c->stream alone
  CK(cudaEventRecord(c->ev_fork, c->stream));
  CK(cudaStreamWaitEvent(c->stream2, c->ev_fork, 0));
  // samples in flight per wave: the path-state arrays hold wave_paths records; a tile of the frame keeps more samples
  // in flight than the whole frame would (3840x2160 whole: 8, one of 8 tiles: 64)
  const int wave_S = (int)std::max<size_t>(1, std::min<size_t>((size_t)c->wave_cap, c->wave_paths / ((size_t)fp.rw * fp.rh)));
  int rc = FSPT_OK;
  for (int done = 0; done < n_samples && !rc;) {
    const int S = std::min(wave_S, n_samples - done);
    if (done > 0 && S != wave_S) {
      // The last, shorter wave splits the rectangle differently (other slice offsets, perhaps one band only), so its
      // bands may touch slices and pixel rows the other stream's band of the previous wave still works on: both streams
      // wait for each other here.  Waves of equal S keep each band on its own stream, slice and rows.
      CK(cudaEventRecord(c->ev_fork, c->stream));
      CK(cudaEventRecord(c->ev_join, c->stream2));
      CK(cudaStreamWaitEvent(c->stream2, c->ev_fork, 0));
      CK(cudaStreamWaitEvent(c->stream, c->ev_join, 0));
    }
    rc = render_wave(c, fp, first_tick + (uint32_t)done, S, c->d_rb.p + done, c->d_rb.p + c->rb_cap + done);
    done += S;
  }
  CK(cudaEventRecord(c->ev_join, c->stream2));  // (also after a failed wave: no work may be left outside c->stream)
  CK(cudaStreamWaitEvent(c->stream, c->ev_join, 0));
  if (rc) return rc;
  CK(cudaEventRecord(c->ev_end, c->stream));
  c->render_timed = true;
  c->next_tick = first_tick + (uint32_t)n_samples;
  c->accum_samples += (uint64_t)n_samples;
  if (!adaptive) c->stats.samples += (uint64_t)n_samples * (uint64_t)fp.rw * (uint64_t)fp.rh;  // (adaptive: d_stats[8])
  return FSPT_OK;
}

int fspt_synchronize(fspt_ctx* ctx) {
  Ctx* c = reinterpret_cast<Ctx*>(ctx);
  if (!c) return FSPT_E_INVALID;
  CK(cudaSetDevice(c->device));
  if (int rc = broadcast_phase2(c)) return rc;  // (joins the atlas thread on the root, see render_wave)
  if (int rc = atlas_join(c)) return rc;
  CK(cudaStreamSynchronize(c->stream));
  CK(cudaStreamSynchronize(c->copy_stream));
  return FSPT_OK;
}

int fspt_resolve(fspt_ctx* ctx, const fspt_post_params* post, uint8_t* rgba8_out) {
  Ctx* c = reinterpret_cast<Ctx*>(ctx);
  if (!c) return FSPT_E_INVALID;
  if (!post || !rgba8_out) return fail(c, FSPT_E_INVALID, "fspt_resolve: NULL argument");
  CK(cudaSetDevice(c->device));
  dim3 blk(32, 8), grd((c->width + 31) / 32, (c->height + 7) / 8);
  const int use_div = c->accum_mode == 1;  // sum mode: every pixel is divided by its own sample count (alpha channel)
  k_post<<<grd, blk, 0, c->stream>>>(c->d_fb.p, c->d_rgba8.p, c->width, c->height, post->exposure, post->saturation,
                                     post->denoise ? 1 : 0, post->max_sigma, post->scale, use_div);
  c->stats.kernel_launches++;
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(rgba8_out, c->d_rgba8.p, (size_t)c->n_pixels * 4, cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  return FSPT_OK;
}

int fspt_read_accum(fspt_ctx* ctx, float* out) {
  Ctx* c = reinterpret_cast<Ctx*>(ctx);
  if (!c || !out) return FSPT_E_INVALID;
  CK(cudaSetDevice(c->device));
  CK(cudaMemcpyAsync(out, c->d_fb.p, (size_t)c->n_pixels * 16, cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  return FSPT_OK;
}

int fspt_write_accum(fspt_ctx* ctx, const float* in, uint32_t next_tick) {
  Ctx* c = reinterpret_cast<Ctx*>(ctx);
  if (!c || !in) return FSPT_E_INVALID;
  CK(cudaSetDevice(c->device));
  CK(cudaMemcpyAsync(c->d_fb.p, in, (size_t)c->n_pixels * 16, cudaMemcpyHostToDevice, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  c->next_tick = next_tick;
  c->accum_samples = next_tick;
  return FSPT_OK;
}

int fspt_set_accum_mode(fspt_ctx* ctx, int32_t mode) {
  Ctx* c = reinterpret_cast<Ctx*>(ctx);
  if (!c || (mode != 0 && mode != 1)) return FSPT_E_INVALID;
  c->accum_mode = mode;
  return FSPT_OK;
}

int fspt_accum_device_ptr(fspt_ctx* ctx, void** dptr, uint64_t* n_floats, uint64_t* n_samples) {
  Ctx* c = reinterpret_cast<Ctx*>(ctx);
  if (!c) return FSPT_E_INVALID;
  CK(cudaSetDevice(c->device));
  CK(cudaStreamSynchronize(c->stream));
  if (dptr) *dptr = c->d_fb.p;
  if (n_floats) *n_floats = (uint64_t)c->n_pixels * 4;
  if (n_samples) *n_samples = c->accum_samples;
  return FSPT_OK;
}

int fspt_set_accum_samples(fspt_ctx* ctx, uint64_t n) {
  Ctx* c = reinterpret_cast<Ctx*>(ctx);
  if (!c) return FSPT_E_INVALID;
  c->accum_samples = n;
  return FSPT_OK;
}

int fspt_set_adaptive(fspt_ctx* ctx, float max_rel_error, int32_t min_samples) {
  Ctx* c = reinterpret_cast<Ctx*>(ctx);
  if (!c) return FSPT_E_INVALID;
  if (!(max_rel_error >= 0.0f) || min_samples < 2)  // (NaN fails the comparison; a variance needs two samples)
    return fail(c, FSPT_E_INVALID, "fspt_set_adaptive: max_rel_error %g must be >= 0 and min_samples %d >= 2",
                (double)max_rel_error, min_samples);
  if (max_rel_error > 0.0f && !c->d_list.p) {
    CK(cudaSetDevice(c->device));
    if (!c->d_m2.p) {
      CK(c->d_m2.fit((size_t)c->n_pixels * sizeof(float)));
      CK(cudaMemsetAsync(c->d_m2.p, 0, (size_t)c->n_pixels * sizeof(float), c->stream));
    }
    CK(c->d_list.fit((size_t)c->n_pixels * sizeof(int)));
  }
  c->adapt_err = max_rel_error;
  c->adapt_min = min_samples;
  return FSPT_OK;
}

int fspt_active_pixels(fspt_ctx* ctx, uint64_t* n_out) {
  Ctx* c = reinterpret_cast<Ctx*>(ctx);
  if (!c || !n_out) return FSPT_E_INVALID;
  if (!(c->adapt_err > 0.0f)) return fail(c, FSPT_E_STATE, "fspt_active_pixels: adaptive sampling is off (fspt_set_adaptive)");
  CK(cudaSetDevice(c->device));
  FrameParams f;
  memset(&f, 0, sizeof f);
  f.width = c->width; f.height = c->height;
  set_rect(f, c->rx0, c->ry0, c->rw, c->rh);
  if (int rc = select_active(c, 0, f, nullptr, 0)) return rc;
  int n = 0;
  CK(cudaMemcpyAsync(&n, band_counts(c, 0) + 8, sizeof n, cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  *n_out = (uint64_t)n;
  return FSPT_OK;
}

int fspt_read_moment(fspt_ctx* ctx, float* out) {
  Ctx* c = reinterpret_cast<Ctx*>(ctx);
  if (!c || !out) return FSPT_E_INVALID;
  if (!c->d_m2.p) return fail(c, FSPT_E_STATE, "fspt_read_moment: adaptive sampling has never been on (fspt_set_adaptive)");
  CK(cudaSetDevice(c->device));
  CK(cudaMemcpyAsync(out, c->d_m2.p, (size_t)c->n_pixels * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  return FSPT_OK;
}

int fspt_write_moment(fspt_ctx* ctx, const float* in) {
  Ctx* c = reinterpret_cast<Ctx*>(ctx);
  if (!c || !in) return FSPT_E_INVALID;
  if (!c->d_m2.p) return fail(c, FSPT_E_STATE, "fspt_write_moment: adaptive sampling has never been on (fspt_set_adaptive)");
  CK(cudaSetDevice(c->device));
  CK(cudaMemcpyAsync(c->d_m2.p, in, (size_t)c->n_pixels * sizeof(float), cudaMemcpyHostToDevice, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  return FSPT_OK;
}

int fspt_debug_primary(fspt_ctx* ctx, const fspt_frame_params* frame, float rand_base_camera, int32_t* index_out,
                       float* t_out, int32_t* count_out, float* pos4_out, float* dir4_out) {
  Ctx* c = reinterpret_cast<Ctx*>(ctx);
  if (!c || !frame) return FSPT_E_INVALID;
  if (!c->has_scene) return fail(c, FSPT_E_STATE, "fspt_debug_primary before fspt_scene_upload");
  CK(cudaSetDevice(c->device));
  const FrameParams fp = make_frame(c, frame, true);  // always the whole frame
  const int P = c->n_pixels;
  {
    int rc0 = stage_rand_bases(c, &rand_base_camera, nullptr, 1);
    if (rc0) return rc0;
  }
  k_camera<<<(P + 255) / 256, 256, 0, c->stream>>>(fp, c->d_rb.p, P, make_fastdiv(1u, (unsigned long long)P), c->ps, c->d_cam_pos.p, c->d_cam_dir.p);
  c->stats.kernel_launches++;
  int rc = set_counts(c, 0, P, 0);
  if (rc) return rc;
  c->ev_trace_used = 0;
  rc = launch_trace(c, 0, band_slice(c, 0), 0, false, true);
  if (rc) return rc;
  CK(cudaStreamSynchronize(c->stream));
  // un-swizzle path slots -> pixels on the host
  std::vector<float4> ro(P), rdv(P);
  std::vector<int> cnt(P);
  CK(cudaMemcpy2D(ro.data(), 16, c->ps.rec + 0, 16 * FSPT_PATH_WORDS, 16, P, cudaMemcpyDeviceToHost));
  CK(cudaMemcpy2D(rdv.data(), 16, c->ps.rec + 1, 16 * FSPT_PATH_WORDS, 16, P, cudaMemcpyDeviceToHost));
  CK(cudaMemcpy(cnt.data(), c->d_count_out.p, (size_t)P * 4, cudaMemcpyDeviceToHost));
  for (int j = 0; j < P; ++j) {
    int x, y;
    if (fp.tiled) {
      const int tiles_x = fp.width >> 3, tile = j >> 5, l = j & 31;
      x = ((tile % tiles_x) << 3) + (l & 7);
      y = ((tile / tiles_x) << 2) + (l >> 3);
    } else { x = j % fp.width; y = j / fp.width; }
    const size_t px = (size_t)y * fp.width + x;
    if (t_out) t_out[px] = ro[j].w;
    if (index_out) memcpy(&index_out[px], &rdv[j].w, 4);
    if (count_out) count_out[px] = cnt[j];
  }
  if (pos4_out) CK(cudaMemcpy(pos4_out, c->d_cam_pos.p, (size_t)P * 16, cudaMemcpyDeviceToHost));
  if (dir4_out) CK(cudaMemcpy(dir4_out, c->d_cam_dir.p, (size_t)P * 16, cudaMemcpyDeviceToHost));
  return pull_stats(c);
}

int fspt_debug_trace(fspt_ctx* ctx, const float* pos4, const float* dir4, int32_t n_rays, int32_t* index_out,
                     float* t_out, int32_t* count_out) {
  Ctx* c = reinterpret_cast<Ctx*>(ctx);
  if (!c || !pos4 || !dir4 || n_rays < 0) return FSPT_E_INVALID;
  if (!c->has_scene) return fail(c, FSPT_E_STATE, "fspt_debug_trace before fspt_scene_upload");
  CK(cudaSetDevice(c->device));
  std::vector<float4> ro, rdv;
  std::vector<int> cnt;
  for (int64_t done = 0; done < n_rays;) {
    const int n = (int)std::min<int64_t>((int64_t)c->wave_paths, n_rays - done);
    CK(cudaMemcpy2DAsync(c->ps.rec + 0, 16 * FSPT_PATH_WORDS, pos4 + 4 * done, 16, 16, n, cudaMemcpyHostToDevice, c->stream));
    CK(cudaMemcpy2DAsync(c->ps.rec + 1, 16 * FSPT_PATH_WORDS, dir4 + 4 * done, 16, 16, n, cudaMemcpyHostToDevice, c->stream));
    int rc = set_counts(c, 0, n, 0);
    if (rc) return rc;
    c->ev_trace_used = 0;
    rc = launch_trace(c, 0, band_slice(c, 0), 0, false, true);
    if (rc) return rc;
    ro.resize(n); rdv.resize(n); cnt.resize(n);
    CK(cudaMemcpy2DAsync(ro.data(), 16, c->ps.rec + 0, 16 * FSPT_PATH_WORDS, 16, n, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaMemcpy2DAsync(rdv.data(), 16, c->ps.rec + 1, 16 * FSPT_PATH_WORDS, 16, n, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaMemcpyAsync(cnt.data(), c->d_count_out.p, (size_t)n * 4, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    for (int i = 0; i < n; ++i) {
      if (t_out) t_out[done + i] = ro[i].w;
      if (index_out) memcpy(&index_out[done + i], &rdv[i].w, 4);
      if (count_out) count_out[done + i] = cnt[i];
    }
    done += n;
  }
  return pull_stats(c);
}

int fspt_debug_last_color(fspt_ctx* ctx, float* out) {
  Ctx* c = reinterpret_cast<Ctx*>(ctx);
  if (!c || !out) return FSPT_E_INVALID;
  CK(cudaSetDevice(c->device));
  CK(cudaMemcpyAsync(out, c->d_last_color.p, (size_t)c->n_pixels * 16, cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  return FSPT_OK;
}

int fspt_debug_math(fspt_ctx* ctx, int32_t fn, const float* x, const float* y, float* out, int32_t n) {
  Ctx* c = reinterpret_cast<Ctx*>(ctx);
  const bool known = (fn >= 0 && fn < FSPT_DEBUG_MATH_CODES) || (fn >= FSPT_DEBUG_MATH_PACKED && fn < FSPT_DEBUG_MATH_PACKED + 4);
  if (!c || !x || !out || n < 0 || !known) return FSPT_E_INVALID;
  CK(cudaSetDevice(c->device));
  DevBuf<float> buf;  // one allocation (x | y | out), released on every path
  const size_t stride = (size_t)n + 1;
  CK(buf.fit(3 * stride * 4));
  float *dx = buf.p, *dy = buf.p + stride, *dout = buf.p + 2 * stride;
  CK(cudaMemcpy(dx, x, (size_t)n * 4, cudaMemcpyHostToDevice));
  if (y) CK(cudaMemcpy(dy, y, (size_t)n * 4, cudaMemcpyHostToDevice)); else CK(cudaMemset(dy, 0, (size_t)n * 4));
  if (n) k_debug_math<<<(n + 255) / 256, 256, 0, c->stream>>>(fn, dx, dy, dout, n);
  CK(cudaStreamSynchronize(c->stream));
  CK(cudaMemcpy(out, dout, (size_t)n * 4, cudaMemcpyDeviceToHost));
  return FSPT_OK;
}

__global__ void __launch_bounds__(256) k_read_bw(const uint4* __restrict__ buf, size_t n16, int iters, unsigned* sink) {
  unsigned acc = 0;
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (int it = 0; it < iters; ++it) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    for (; i + 3 * stride < n16; i += 4 * stride) {  // four independent loads in flight per thread
      const uint4 a = __ldcg(buf + i), b = __ldcg(buf + i + stride), c2 = __ldcg(buf + i + 2 * stride), d = __ldcg(buf + i + 3 * stride);
      acc ^= a.x ^ a.y ^ a.z ^ a.w ^ b.x ^ b.y ^ b.z ^ b.w ^ c2.x ^ c2.y ^ c2.z ^ c2.w ^ d.x ^ d.y ^ d.z ^ d.w;
    }
    for (; i < n16; i += stride) { const uint4 a = __ldcg(buf + i); acc ^= a.x ^ a.y ^ a.z ^ a.w; }
  }
  if (acc == 0x9e3779b9u) *sink = acc;  // keeps the loads alive
}

int fspt_debug_read_bandwidth(fspt_ctx* ctx, uint64_t bytes, int32_t iters, double* gb_per_s_out) {
  Ctx* c = reinterpret_cast<Ctx*>(ctx);
  if (!c || !gb_per_s_out || bytes < 4096 || iters < 1) return FSPT_E_INVALID;
  CK(cudaSetDevice(c->device));
  DevBuf<uint4> buf;
  DevBuf<unsigned> sink;
  const size_t n16 = (size_t)bytes / 16;
  CK(buf.fit(n16 * 16));
  CK(sink.fit(4));
  CK(cudaMemsetAsync(buf.p, 1, n16 * 16, c->stream));
  Event e0, e1;
  CK(e0.create(cudaEventDefault)); CK(e1.create(cudaEventDefault));
  const int blocks = c->sm_count * 8;
  k_read_bw<<<blocks, 256, 0, c->stream>>>(buf.p, n16, 1, sink.p);  // warm-up: brings the buffer into L2 when it fits
  CK(cudaEventRecord(e0, c->stream));
  k_read_bw<<<blocks, 256, 0, c->stream>>>(buf.p, n16, iters, sink.p);
  CK(cudaEventRecord(e1, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  float ms = 0.0f;
  CK(cudaEventElapsedTime(&ms, e0, e1));
  *gb_per_s_out = (double)n16 * 16.0 * iters / (ms * 1e-3) / 1e9;
  return FSPT_OK;
}

int fspt_set_tile(fspt_ctx* ctx, int32_t x0, int32_t y0, int32_t w, int32_t h) {
  Ctx* c = reinterpret_cast<Ctx*>(ctx);
  if (!c) return FSPT_E_INVALID;
  if (w <= 0 || h <= 0 || x0 < 0 || y0 < 0 || (int64_t)x0 + w > c->width || (int64_t)y0 + h > c->height)
    return fail(c, FSPT_E_INVALID, "fspt_set_tile: rectangle %d,%d %dx%d is not inside the %dx%d frame", x0, y0, w, h, c->width, c->height);
  c->rx0 = x0; c->ry0 = y0; c->rw = w; c->rh = h;
  return FSPT_OK;
}

int fspt_comm_unique_id(uint8_t* id_out) {
  Ctx* c = nullptr;
  if (!id_out) return FSPT_E_INVALID;
  NcclApi* N = nccl_api();
  if (!N->error.empty()) return fail(c, FSPT_E_NCCL, "%s", N->error.c_str());
  ncclUniqueId id;
  NK(N->GetUniqueId(&id));
  static_assert(sizeof(id) == FSPT_COMM_ID_BYTES, "ncclUniqueId size");
  memcpy(id_out, &id, sizeof id);
  return FSPT_OK;
}

int fspt_comm_init(fspt_ctx* ctx, const uint8_t* id_bytes, int32_t rank, int32_t world) {
  Ctx* c = reinterpret_cast<Ctx*>(ctx);
  if (!c || !id_bytes || world < 1 || rank < 0 || rank >= world) return FSPT_E_INVALID;
  NcclApi* N = nccl_api();
  if (!N->error.empty()) return fail(c, FSPT_E_NCCL, "%s", N->error.c_str());
  CK(cudaSetDevice(c->device));
  comm_free(c);
  ncclUniqueId id;
  memcpy(&id, id_bytes, sizeof id);
  NK(N->CommInitRank(&c->comm, world, id, rank));
  c->comm_rank = rank; c->comm_world = world;
  CK(c->d_hdr.fit(512));  // [0, 256) geometry header, [256, 512) atlas header
  return FSPT_OK;
}

int fspt_comm_destroy(fspt_ctx* ctx) {
  Ctx* c = reinterpret_cast<Ctx*>(ctx);
  if (!c) return FSPT_E_INVALID;
  CK(cudaSetDevice(c->device));
  CK(cudaStreamSynchronize(c->stream));
  comm_free(c);
  return FSPT_OK;
}

// sum of the accumulation targets of every rank -> root's target, in place, on the context's stream (ordered after the
// render kernels already enqueued, no host synchronisation).  In sum mode the alpha channel carries every pixel's sample
// count, so tiles, sample sets and unequal shards all resolve correctly on the root.
int fspt_reduce_accum(fspt_ctx* ctx, int32_t root) {
  Ctx* c = reinterpret_cast<Ctx*>(ctx);
  if (!c) return FSPT_E_INVALID;
  if (!c->comm) return fail(c, FSPT_E_STATE, "fspt_reduce_accum before fspt_comm_init");
  if (root < 0 || root >= c->comm_world) return fail(c, FSPT_E_INVALID, "fspt_reduce_accum: root %d of %d ranks", root, c->comm_world);
  if (c->accum_mode != 1) return fail(c, FSPT_E_STATE, "fspt_reduce_accum needs the sum accumulation mode (fspt_set_accum_mode(ctx, 1))");
  CK(cudaSetDevice(c->device));
  if (int rc = broadcast_phase2(c)) return rc;  // (a rank that rendered nothing since the broadcast)
  NcclApi* N = nccl_api();
  CK(cudaEventRecord(c->ev_red0, c->stream));
  NK(N->Reduce(c->d_fb.p, c->d_fb.p, (size_t)c->n_pixels * 4, ncclFloat32, ncclSum, root, c->comm, c->stream));
  CK(cudaEventRecord(c->ev_red1, c->stream));
  c->reduce_timed = true;
  c->stats.kernel_launches++;
  return FSPT_OK;
}

int fspt_scene_broadcast(fspt_ctx* ctx, int32_t root) {
  Ctx* c = reinterpret_cast<Ctx*>(ctx);
  if (!c) return FSPT_E_INVALID;
  if (!c->comm) return fail(c, FSPT_E_STATE, "fspt_scene_broadcast before fspt_comm_init");
  if (root < 0 || root >= c->comm_world) return fail(c, FSPT_E_INVALID, "fspt_scene_broadcast: root %d of %d ranks", root, c->comm_world);
  const bool is_root = c->comm_rank == root;
  if (is_root && !c->has_scene) return fail(c, FSPT_E_STATE, "fspt_scene_broadcast: the root has no scene (fspt_scene_upload first)");
  CK(cudaSetDevice(c->device));
  int rc;
  if ((rc = broadcast_phase2(c))) return rc;  // (a previous broadcast nobody rendered from)
  if (!is_root && (rc = atlas_join(c))) return rc;
  NcclApi* N = nccl_api();
  SceneHeader h;
  memset(&h, 0, sizeof h);
  static_assert(sizeof(SceneHeader) <= 256, "header buffer");
  if (is_root) {
    h.scene = c->info;
    h.magic = 0x46535054;
    CK(cudaMemcpyAsync(c->d_hdr.p, &h, sizeof h, cudaMemcpyHostToDevice, c->stream));
  } else {
    CK(cudaStreamSynchronize(c->stream));  // nothing of the previous scene may still be in flight
    CK(cudaStreamSynchronize(c->copy_stream));
  }
  NK(N->Broadcast(c->d_hdr.p, c->d_hdr.p, sizeof h, ncclUint8, root, c->comm, c->stream));
  if (!is_root) {
    CK(cudaMemcpyAsync(&h, c->d_hdr.p, sizeof h, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    if (h.magic != 0x46535054) return fail(c, FSPT_E_NCCL, "fspt_scene_broadcast: bad header from rank %d", root);
  }
  const SceneInfo& si = h.scene;
  const size_t env_pitch = (size_t)si.env_w * 4, env_bytes = env_pitch * si.env_h;
  CK(c->d_lin_env.fit(env_bytes));
  uint8_t* lin = c->d_lin_env.p;
  if (is_root) {
    CK(cudaMemcpy2DFromArrayAsync(lin, env_pitch, c->env.arr, 0, 0, env_pitch, si.env_h, cudaMemcpyDeviceToDevice, c->stream));
  } else {
    // storage on the receiving side: same reuse rules as fspt_scene_upload
    c->has_scene = false;
    if ((rc = fit_scene(c, si))) return rc;
  }
  NK(N->GroupStart());
  NK(N->Broadcast(c->d_nodes.p, c->d_nodes.p, si.bytes_nodes, ncclUint8, root, c->comm, c->stream));
  NK(N->Broadcast(c->d_tris.p, c->d_tris.p, si.bytes_tris, ncclUint8, root, c->comm, c->stream));
  NK(N->Broadcast(c->d_shade.p, c->d_shade.p, si.bytes_shade, ncclUint8, root, c->comm, c->stream));
  NK(N->Broadcast(c->d_bins.p, c->d_bins.p, si.bytes_bins, ncclUint8, root, c->comm, c->stream));
  NK(N->Broadcast(lin, lin, env_bytes, ncclUint8, root, c->comm, c->stream));
  NK(N->GroupEnd());
  c->stats.kernel_launches += 6;
  if (!is_root) {
    CK(cudaMemcpy2DToArrayAsync(c->env.arr, 0, 0, lin, env_pitch, env_pitch, si.env_h, cudaMemcpyDeviceToDevice, c->stream));
    if ((rc = publish_scene(c, si))) return rc;
    c->has_scene = true;
  }
  CK(cudaEventRecord(c->ev_bcast, c->stream));
  c->bcast_pending_root = root;  // phase 2: the atlas, behind the next primary traversal launch
  return FSPT_OK;
}

int fspt_set_param(fspt_ctx* ctx, int32_t key, int32_t value) {
  Ctx* c = reinterpret_cast<Ctx*>(ctx);
  if (!c) return FSPT_E_INVALID;
  switch (key) {
    case FSPT_PARAM_ANYHIT: c->anyhit = value ? 1 : 0; return FSPT_OK;
    case FSPT_PARAM_MAX_REFRACTIONS:
      if (value < 0 || value > 30000) return fail(c, FSPT_E_INVALID, "max_refractions out of range");
      c->max_refractions = value; return FSPT_OK;
    case FSPT_PARAM_SANITIZE_NAN: c->sanitize = value ? 1 : 0; return FSPT_OK;
  }
  return fail(c, FSPT_E_INVALID, "fspt_set_param: unknown key %d", key);
}

int fspt_get_stats(fspt_ctx* ctx, fspt_stats* out) {
  Ctx* c = reinterpret_cast<Ctx*>(ctx);
  if (!c || !out) return FSPT_E_INVALID;
  CK(cudaSetDevice(c->device));
  CK(cudaStreamSynchronize(c->stream));
  int rc = pull_stats(c);
  if (rc) return rc;
  float ms = 0.0f;
  if (c->render_timed && cudaEventElapsedTime(&ms, c->ev_begin, c->ev_end) == cudaSuccess) c->stats.render_ms = ms;
  double tr = 0.0, sh = 0.0, pr = 0.0;
  for (size_t i = 0; i + 1 < c->ev_trace_used; i += 2) {
    float t = 0.0f;
    if (cudaEventElapsedTime(&t, c->ev_trace[i], c->ev_trace[i + 1]) != cudaSuccess) continue;
    const int tag = c->ev_tag[i / 2];
    (tag == 1 ? sh : tr) += t;
    if (tag == 2) pr += t;
  }
  c->stats.shade_ms = sh;
  c->stats.primary_trace_ms = pr;
  c->stats.reduce_ms = 0.0;
  if (c->reduce_timed && cudaEventElapsedTime(&ms, c->ev_red0, c->ev_red1) == cudaSuccess) c->stats.reduce_ms = ms;
  (void)cudaGetLastError();  // event queries must not leave a sticky status for the next launch check
  c->stats.trace_ms = tr;
  *out = c->stats;
  out->samples += c->adaptive_samples;
  out->kernel_launches += c->atlas_launches.load();
  return FSPT_OK;
}

}  // extern "C"
