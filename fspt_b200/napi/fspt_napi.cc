// fspt_napi.cc -- thin N-API addon over the C ABI (include/fspt_b200.h) so that a Node.js host can drive the
// B200 path exactly where main.js drives WebGL.  NOT compiled in this image (no Node toolchain / node_api.h; see
// INTEGRATION.md for the build line).  Every export maps 1:1 to a C-ABI call; typed arrays are borrowed for the
// duration of the call, like texImage2D does (main.js:412-437).
//
//   const fspt = require('./build/Release/fspt_napi.node');
//   const ctx = fspt.create(width, height, device);
//   fspt.sceneUpload(ctx, {bvh: Float32Array, triangles, materials, normals, uvs, atlas: Uint8Array,
//                          env: Uint8Array, radianceBins: Uint16Array, atlasRes, atlasLayers, envWidth, envHeight});
//   fspt.render(ctx, {eye, dir, fovScale, lensFeatures, envTheta}, firstTick, randBaseCamera, randBaseTracer);
//   const rgba8 = fspt.resolve(ctx, {exposure, saturation, maxSigma, scale, denoise});
// Multi-GPU (one process per GPU, see main_multi.mjs): fspt.commUniqueId() / commInit(ctx, id, rank, world) /
//   sceneBroadcast(ctx, root) / setTile(ctx, x0, y0, w, h) / setAccumMode(ctx, 1) / reduceAccum(ctx, root).
// Adaptive sampling (sum mode): setAdaptive(ctx, maxRelError, minSamples) / activePixels(ctx) / readMoment(ctx, w, h) /
//   writeMoment(ctx, Float32Array, w, h).
#include <node_api.h>

#include <cstring>
#include <string>
#include <vector>

#include "../../include/fspt_b200.h"

namespace {

#define NAPI_OK(call)                                             \
  do {                                                            \
    if ((call) != napi_ok) {                                      \
      napi_throw_error(env, nullptr, "N-API call failed: " #call); \
      return nullptr;                                             \
    }                                                             \
  } while (0)

napi_value Throw(napi_env env, fspt_ctx* ctx, int rc) {  // non-zero status -> thrown JS Error (INTEGRATION.md)
  std::string msg = "fspt error " + std::to_string(rc) + ": " + fspt_last_error(ctx);
  napi_throw_error(env, nullptr, msg.c_str());
  return nullptr;
}

fspt_ctx* Unwrap(napi_env env, napi_value v) {
  void* p = nullptr;
  napi_get_value_external(env, v, &p);
  return static_cast<fspt_ctx*>(p);
}

template <class T>
T* TypedData(napi_env env, napi_value obj, const char* key, size_t* len) {
  napi_value v;
  bool has = false;
  napi_has_named_property(env, obj, key, &has);
  if (!has) return nullptr;
  napi_get_named_property(env, obj, key, &v);
  napi_typedarray_type type;
  void* data = nullptr;
  napi_value ab;
  size_t off;
  if (napi_get_typedarray_info(env, v, &type, len, &data, &ab, &off) != napi_ok) return nullptr;
  return static_cast<T*>(data);
}

double NumProp(napi_env env, napi_value obj, const char* key, double dflt) {
  napi_value v;
  bool has = false;
  napi_has_named_property(env, obj, key, &has);
  if (!has) return dflt;
  napi_get_named_property(env, obj, key, &v);
  double d = dflt;
  napi_get_value_double(env, v, &d);
  return d;
}

void Vec(napi_env env, napi_value obj, const char* key, float* out, int n) {
  napi_value arr, e;
  napi_get_named_property(env, obj, key, &arr);
  for (int i = 0; i < n; ++i) {
    double d = 0;
    napi_get_element(env, arr, i, &e);
    napi_get_value_double(env, e, &d);  // the reference passes strings for some uniforms; coerce in JS first
    out[i] = (float)d;
  }
}

void Finalize(napi_env, void* data, void*) { fspt_destroy(static_cast<fspt_ctx*>(data)); }

napi_value Create(napi_env env, napi_callback_info info) {
  size_t argc = 3;
  napi_value argv[3];
  NAPI_OK(napi_get_cb_info(env, info, &argc, argv, nullptr, nullptr));
  int32_t w = 0, h = 0, dev = 0;
  napi_get_value_int32(env, argv[0], &w);
  napi_get_value_int32(env, argv[1], &h);
  if (argc > 2) napi_get_value_int32(env, argv[2], &dev);
  fspt_ctx* ctx = nullptr;
  int rc = fspt_create(&ctx, w, h, dev);
  if (rc) return Throw(env, nullptr, rc);
  napi_value ext;
  NAPI_OK(napi_create_external(env, ctx, Finalize, nullptr, &ext));
  return ext;
}

// sceneUpload(ctx, scene[, 1]): a third argument of 1 selects fspt_scene_upload_async -- the host keeps scene.atlas
// alive and untouched until sceneUploadWait(ctx) (typed arrays are borrowed, not copied).
napi_value SceneUpload(napi_env env, napi_callback_info info) {
  size_t argc = 3;
  napi_value argv[3];
  NAPI_OK(napi_get_cb_info(env, info, &argc, argv, nullptr, nullptr));
  int32_t async_atlas = 0;
  if (argc > 2) napi_get_value_int32(env, argv[2], &async_atlas);
  fspt_ctx* ctx = Unwrap(env, argv[0]);
  fspt_scene_desc d;
  std::memset(&d, 0, sizeof d);
  size_t n = 0, nb = 0, nt = 0, nbins = 0;
  d.bvh = TypedData<float>(env, argv[1], "bvh", &nb);
  d.triangles = TypedData<float>(env, argv[1], "triangles", &nt);
  d.materials = TypedData<float>(env, argv[1], "materials", &n);
  d.normals = TypedData<float>(env, argv[1], "normals", &n);
  d.uvs = TypedData<float>(env, argv[1], "uvs", &n);
  d.lights = TypedData<float>(env, argv[1], "lights", &n);
  d.n_light_triangles = d.lights ? (int32_t)(n / 9) : 0;
  d.light_ranges = TypedData<float>(env, argv[1], "lightRanges", &n);
  d.n_light_ranges = d.light_ranges ? (int32_t)(n / 2) : 0;
  d.atlas = TypedData<uint8_t>(env, argv[1], "atlas", &n);
  d.env = TypedData<uint8_t>(env, argv[1], "env", &n);
  d.radiance_bins = TypedData<uint16_t>(env, argv[1], "radianceBins", &nbins);
  d.n_nodes = (int32_t)(nb / 9);
  d.n_triangles = (int32_t)(nt / 9);
  d.atlas_res = (int32_t)NumProp(env, argv[1], "atlasRes", 0);
  d.atlas_layers = (int32_t)NumProp(env, argv[1], "atlasLayers", 0);
  d.env_width = (int32_t)NumProp(env, argv[1], "envWidth", 0);
  d.env_height = (int32_t)NumProp(env, argv[1], "envHeight", 0);
  d.env_bins = (int32_t)(nbins / 4);
  d.leaf_size = (int32_t)NumProp(env, argv[1], "leafSize", 4);
  int rc = async_atlas ? fspt_scene_upload_async(ctx, &d) : fspt_scene_upload(ctx, &d);
  if (rc) return Throw(env, ctx, rc);
  return nullptr;
}

// hostRegister(typedArray) / hostUnregister(typedArray): page-lock the array's backing store in place (fspt_host_register);
// uploads then DMA a page-locked atlas / env from where it lies.  The host must keep the array alive while registered.
napi_value HostRegister(napi_env env, napi_callback_info info) {
  size_t argc = 1;
  napi_value argv[1];
  NAPI_OK(napi_get_cb_info(env, info, &argc, argv, nullptr, nullptr));
  napi_typedarray_type t;
  size_t n = 0, off = 0;
  void* data = nullptr;
  napi_value ab;
  NAPI_OK(napi_get_typedarray_info(env, argv[0], &t, &n, &data, &ab, &off));
  const size_t elem = (t == napi_float32_array || t == napi_int32_array || t == napi_uint32_array) ? 4
                      : (t == napi_uint16_array || t == napi_int16_array) ? 2 : (t == napi_float64_array) ? 8 : 1;
  int r = fspt_host_register(data, (uint64_t)(n * elem));
  if (r) return Throw(env, nullptr, r);
  return nullptr;
}
napi_value HostUnregister(napi_env env, napi_callback_info info) {
  size_t argc = 1;
  napi_value argv[1];
  NAPI_OK(napi_get_cb_info(env, info, &argc, argv, nullptr, nullptr));
  napi_typedarray_type t;
  size_t n = 0, off = 0;
  void* data = nullptr;
  napi_value ab;
  NAPI_OK(napi_get_typedarray_info(env, argv[0], &t, &n, &data, &ab, &off));
  int r = fspt_host_unregister(data);
  if (r) return Throw(env, nullptr, r);
  return nullptr;
}

napi_value SceneUploadWait(napi_env env, napi_callback_info info) {
  size_t argc = 1;
  napi_value argv[1];
  NAPI_OK(napi_get_cb_info(env, info, &argc, argv, nullptr, nullptr));
  fspt_ctx* ctx = Unwrap(env, argv[0]);
  int r = fspt_scene_upload_wait(ctx);
  if (r) return Throw(env, ctx, r);
  return nullptr;
}

void Frame(napi_env env, napi_value obj, fspt_frame_params* f) {
  Vec(env, obj, "eye", f->eye, 3);
  Vec(env, obj, "dir", f->dir, 3);
  Vec(env, obj, "lensFeatures", f->lens_features, 2);
  f->fov_scale = (float)NumProp(env, obj, "fovScale", 0.5);
  f->env_theta = (float)NumProp(env, obj, "envTheta", 0.0);
}

napi_value Render(napi_env env, napi_callback_info info) {
  size_t argc = 5;
  napi_value argv[5];
  NAPI_OK(napi_get_cb_info(env, info, &argc, argv, nullptr, nullptr));
  fspt_ctx* ctx = Unwrap(env, argv[0]);
  fspt_frame_params f;
  Frame(env, argv[1], &f);
  uint32_t first = 0;
  napi_get_value_uint32(env, argv[2], &first);
  napi_typedarray_type t;
  size_t n1 = 0, n2 = 0, off;
  void *rc = nullptr, *rt = nullptr;
  napi_value ab;
  NAPI_OK(napi_get_typedarray_info(env, argv[3], &t, &n1, &rc, &ab, &off));
  NAPI_OK(napi_get_typedarray_info(env, argv[4], &t, &n2, &rt, &ab, &off));
  int r = fspt_render(ctx, &f, first, (int32_t)(n1 < n2 ? n1 : n2), static_cast<float*>(rc), static_cast<float*>(rt));
  if (r) return Throw(env, ctx, r);
  return nullptr;
}

napi_value Clear(napi_env env, napi_callback_info info) {
  size_t argc = 1;
  napi_value argv[1];
  NAPI_OK(napi_get_cb_info(env, info, &argc, argv, nullptr, nullptr));
  fspt_ctx* ctx = Unwrap(env, argv[0]);
  int r = fspt_clear(ctx);
  if (r) return Throw(env, ctx, r);
  return nullptr;
}

napi_value Resolve(napi_env env, napi_callback_info info) {
  size_t argc = 4;
  napi_value argv[4];
  NAPI_OK(napi_get_cb_info(env, info, &argc, argv, nullptr, nullptr));
  fspt_ctx* ctx = Unwrap(env, argv[0]);
  fspt_post_params p;
  p.exposure = (float)NumProp(env, argv[1], "exposure", 1.0);
  p.saturation = (float)NumProp(env, argv[1], "saturation", 1.0);
  p.max_sigma = (float)NumProp(env, argv[1], "maxSigma", 2.0);
  p.scale = (float)NumProp(env, argv[1], "scale", 1.0);
  p.denoise = (int32_t)NumProp(env, argv[1], "denoise", 0);
  int32_t w = 0, h = 0;
  napi_get_value_int32(env, argv[2], &w);
  napi_get_value_int32(env, argv[3], &h);
  void* data = nullptr;
  napi_value ab, out;
  NAPI_OK(napi_create_arraybuffer(env, (size_t)w * h * 4, &data, &ab));
  int r = fspt_resolve(ctx, &p, static_cast<uint8_t*>(data));
  if (r) return Throw(env, ctx, r);
  NAPI_OK(napi_create_typedarray(env, napi_uint8_clamped_array, (size_t)w * h * 4, ab, 0, &out));
  return out;
}

napi_value ReadAccum(napi_env env, napi_callback_info info) {
  size_t argc = 3;
  napi_value argv[3];
  NAPI_OK(napi_get_cb_info(env, info, &argc, argv, nullptr, nullptr));
  fspt_ctx* ctx = Unwrap(env, argv[0]);
  int32_t w = 0, h = 0;
  napi_get_value_int32(env, argv[1], &w);
  napi_get_value_int32(env, argv[2], &h);
  void* data = nullptr;
  napi_value ab, out;
  NAPI_OK(napi_create_arraybuffer(env, (size_t)w * h * 16, &data, &ab));
  int r = fspt_read_accum(ctx, static_cast<float*>(data));
  if (r) return Throw(env, ctx, r);
  NAPI_OK(napi_create_typedarray(env, napi_float32_array, (size_t)w * h * 4, ab, 0, &out));
  return out;
}

napi_value BvhBuild(napi_env env, napi_callback_info info) {  // new BVH(triangles, 4) + serializeTree + flatten
  size_t argc = 1;
  napi_value argv[1];
  NAPI_OK(napi_get_cb_info(env, info, &argc, argv, nullptr, nullptr));
  napi_typedarray_type t;
  size_t n = 0, off;
  void* verts = nullptr;
  napi_value ab;
  NAPI_OK(napi_get_typedarray_info(env, argv[0], &t, &n, &verts, &ab, &off));  // Float64Array, 9 per triangle
  const int32_t T = (int32_t)(n / 9);
  void *nodes = nullptr, *order = nullptr;
  napi_value nab, oab, res, nodesArr, orderArr, v;
  NAPI_OK(napi_create_arraybuffer(env, (size_t)(2 * T + 1) * 36, &nodes, &nab));
  NAPI_OK(napi_create_arraybuffer(env, (size_t)T * 4, &order, &oab));
  int32_t nn = 0, depth = 0;
  int rc = fspt_bvh_build(static_cast<double*>(verts), T, 4, static_cast<float*>(nodes), static_cast<int32_t*>(order), &nn, &depth, 0);
  if (rc) return Throw(env, nullptr, rc);
  NAPI_OK(napi_create_typedarray(env, napi_float32_array, (size_t)nn * 9, nab, 0, &nodesArr));
  NAPI_OK(napi_create_typedarray(env, napi_int32_array, (size_t)T, oab, 0, &orderArr));
  NAPI_OK(napi_create_object(env, &res));
  napi_set_named_property(env, res, "bvh", nodesArr);
  napi_set_named_property(env, res, "order", orderArr);
  napi_create_int32(env, depth, &v);
  napi_set_named_property(env, res, "depth", v);
  return res;
}

// ---- multi-GPU: one Node process (or worker) per GPU; the collectives run inside libfspt_b200.so over NCCL ---------
int32_t Int32Arg(napi_env env, napi_value v) { int32_t x = 0; napi_get_value_int32(env, v, &x); return x; }

napi_value SetTile(napi_env env, napi_callback_info info) {  // setTile(ctx, x0, y0, w, h)
  size_t argc = 5;
  napi_value argv[5];
  NAPI_OK(napi_get_cb_info(env, info, &argc, argv, nullptr, nullptr));
  fspt_ctx* ctx = Unwrap(env, argv[0]);
  int r = fspt_set_tile(ctx, Int32Arg(env, argv[1]), Int32Arg(env, argv[2]), Int32Arg(env, argv[3]), Int32Arg(env, argv[4]));
  if (r) return Throw(env, ctx, r);
  return nullptr;
}

napi_value SetAccumMode(napi_env env, napi_callback_info info) {  // setAccumMode(ctx, 0 | 1)
  size_t argc = 2;
  napi_value argv[2];
  NAPI_OK(napi_get_cb_info(env, info, &argc, argv, nullptr, nullptr));
  fspt_ctx* ctx = Unwrap(env, argv[0]);
  int r = fspt_set_accum_mode(ctx, Int32Arg(env, argv[1]));
  if (r) return Throw(env, ctx, r);
  return nullptr;
}

napi_value CommUniqueId(napi_env env, napi_callback_info) {  // -> Uint8Array(128); rank 0 calls it and ships it
  void* data = nullptr;
  napi_value ab, out;
  NAPI_OK(napi_create_arraybuffer(env, FSPT_COMM_ID_BYTES, &data, &ab));
  int r = fspt_comm_unique_id(static_cast<uint8_t*>(data));
  if (r) return Throw(env, nullptr, r);
  NAPI_OK(napi_create_typedarray(env, napi_uint8_array, FSPT_COMM_ID_BYTES, ab, 0, &out));
  return out;
}

napi_value CommInit(napi_env env, napi_callback_info info) {  // commInit(ctx, idUint8Array, rank, world)
  size_t argc = 4;
  napi_value argv[4];
  NAPI_OK(napi_get_cb_info(env, info, &argc, argv, nullptr, nullptr));
  fspt_ctx* ctx = Unwrap(env, argv[0]);
  napi_typedarray_type t;
  size_t n = 0, off;
  void* id = nullptr;
  napi_value ab;
  NAPI_OK(napi_get_typedarray_info(env, argv[1], &t, &n, &id, &ab, &off));
  if (n < FSPT_COMM_ID_BYTES) { napi_throw_error(env, nullptr, "commInit: the id must hold 128 bytes"); return nullptr; }
  int r = fspt_comm_init(ctx, static_cast<uint8_t*>(id), Int32Arg(env, argv[2]), Int32Arg(env, argv[3]));
  if (r) return Throw(env, ctx, r);
  return nullptr;
}

napi_value ReduceAccum(napi_env env, napi_callback_info info) {  // reduceAccum(ctx, root)
  size_t argc = 2;
  napi_value argv[2];
  NAPI_OK(napi_get_cb_info(env, info, &argc, argv, nullptr, nullptr));
  fspt_ctx* ctx = Unwrap(env, argv[0]);
  int r = fspt_reduce_accum(ctx, Int32Arg(env, argv[1]));
  if (r) return Throw(env, ctx, r);
  return nullptr;
}

napi_value SceneBroadcast(napi_env env, napi_callback_info info) {  // sceneBroadcast(ctx, root)
  size_t argc = 2;
  napi_value argv[2];
  NAPI_OK(napi_get_cb_info(env, info, &argc, argv, nullptr, nullptr));
  fspt_ctx* ctx = Unwrap(env, argv[0]);
  int r = fspt_scene_broadcast(ctx, Int32Arg(env, argv[1]));
  if (r) return Throw(env, ctx, r);
  return nullptr;
}

// ---- adaptive sampling (fspt_set_adaptive): render until the pixels' means have converged ----------------------------
napi_value SetAdaptive(napi_env env, napi_callback_info info) {  // setAdaptive(ctx, maxRelError, minSamples)
  size_t argc = 3;
  napi_value argv[3];
  NAPI_OK(napi_get_cb_info(env, info, &argc, argv, nullptr, nullptr));
  fspt_ctx* ctx = Unwrap(env, argv[0]);
  double err = 0;
  napi_get_value_double(env, argv[1], &err);
  int r = fspt_set_adaptive(ctx, (float)err, argc > 2 ? Int32Arg(env, argv[2]) : 16);
  if (r) return Throw(env, ctx, r);
  return nullptr;
}

napi_value ActivePixels(napi_env env, napi_callback_info info) {  // activePixels(ctx) -> pixels the next wave renders
  size_t argc = 1;
  napi_value argv[1];
  NAPI_OK(napi_get_cb_info(env, info, &argc, argv, nullptr, nullptr));
  fspt_ctx* ctx = Unwrap(env, argv[0]);
  uint64_t n = 0;
  int r = fspt_active_pixels(ctx, &n);
  if (r) return Throw(env, ctx, r);
  napi_value out;
  NAPI_OK(napi_create_int32(env, (int32_t)n, &out));  // (fspt_create bounds a frame by 2^27 pixels)
  return out;
}

napi_value ReadMoment(napi_env env, napi_callback_info info) {  // readMoment(ctx, w, h) -> Float32Array(w * h)
  size_t argc = 3;
  napi_value argv[3];
  NAPI_OK(napi_get_cb_info(env, info, &argc, argv, nullptr, nullptr));
  fspt_ctx* ctx = Unwrap(env, argv[0]);
  const size_t n = (size_t)Int32Arg(env, argv[1]) * (size_t)Int32Arg(env, argv[2]);
  void* data = nullptr;
  napi_value ab, out;
  NAPI_OK(napi_create_arraybuffer(env, n * 4, &data, &ab));
  int r = fspt_read_moment(ctx, static_cast<float*>(data));
  if (r) return Throw(env, ctx, r);
  NAPI_OK(napi_create_typedarray(env, napi_float32_array, n, ab, 0, &out));
  return out;
}

napi_value WriteMoment(napi_env env, napi_callback_info info) {  // writeMoment(ctx, Float32Array(w * h), w, h)
  size_t argc = 4;
  napi_value argv[4];
  NAPI_OK(napi_get_cb_info(env, info, &argc, argv, nullptr, nullptr));
  fspt_ctx* ctx = Unwrap(env, argv[0]);
  napi_typedarray_type t;
  size_t n = 0, off;
  void* data = nullptr;
  napi_value ab;
  NAPI_OK(napi_get_typedarray_info(env, argv[1], &t, &n, &data, &ab, &off));
  if (t != napi_float32_array || n < (size_t)Int32Arg(env, argv[2]) * (size_t)Int32Arg(env, argv[3])) {
    napi_throw_error(env, nullptr, "writeMoment: needs a Float32Array of w * h values");
    return nullptr;
  }
  int r = fspt_write_moment(ctx, static_cast<const float*>(data));
  if (r) return Throw(env, ctx, r);
  return nullptr;
}

napi_value Init(napi_env env, napi_value exports) {
  const struct { const char* name; napi_callback fn; } fns[] = {
      {"create", Create}, {"sceneUpload", SceneUpload}, {"sceneUploadWait", SceneUploadWait},
      {"hostRegister", HostRegister}, {"hostUnregister", HostUnregister}, {"render", Render}, {"clear", Clear},
      {"resolve", Resolve}, {"readAccum", ReadAccum}, {"bvhBuild", BvhBuild},
      {"setTile", SetTile}, {"setAccumMode", SetAccumMode}, {"commUniqueId", CommUniqueId}, {"commInit", CommInit},
      {"reduceAccum", ReduceAccum}, {"sceneBroadcast", SceneBroadcast}, {"setAdaptive", SetAdaptive},
      {"activePixels", ActivePixels}, {"readMoment", ReadMoment}, {"writeMoment", WriteMoment}};
  for (auto& f : fns) {
    napi_value fn;
    napi_create_function(env, f.name, NAPI_AUTO_LENGTH, f.fn, nullptr, &fn);
    napi_set_named_property(env, exports, f.name, fn);
  }
  return exports;
}

}  // namespace

NAPI_MODULE(NODE_GYP_MODULE_NAME, Init)
