// camera.cuh -- the sin-hash RNG of the reference shaders and thin-lens ray generation (camera.fs:19-46).
#pragma once
#include "device_common.cuh"
#include "dm_math.cuh"

// rnd(), tracer.fs:181 / camera.fs:19
// (kept out of line: the shading kernel calls it ~8 times per vertex)
__device__ __noinline__ float sin_hash(float seed) { return fractf(dm::sinf_(seed) * 43758.5453123f); }
__device__ __forceinline__ float rnd(float& seed) {
  seed += 0.211324865405187f;
  return sin_hash(seed);
}

// camera.fs main, :37-46, for path slot p.  slot = pixel * S + sample: the S samples of one pixel sit in adjacent
// slots (adjacent lanes), so their primary rays, hit records and texel footprints coincide and are served once per
// warp instead of once per sample.
// LIST (adaptive sampling): j indexes `list`, which holds the slots of the pixels this wave renders (adaptive.cuh).
template <bool LIST = false>
__device__ __forceinline__ void camera_ray(const FrameParams& f, const float* __restrict__ rb_cam, const FastDiv& div_s, int p,
                                           v3& o, v3& d, int& x, int& y, const int* __restrict__ list = nullptr) {
  const int j = (int)fast_div((unsigned)p, div_s), s = p - j * (int)div_s.d;  // div_s: by the samples per wave
  path_to_pixel(f, LIST ? list[j] : j, x, y);  // inside the context's rectangle; gl_FragCoord is the frame pixel
  const float resx = (float)f.width, resy = (float)f.height;
  const float fx = (float)(x + f.rx0) + 0.5f, fy = (float)(y + f.ry0) + 0.5f;  // gl_FragCoord
  const float uvx = (fx / resx) * 2.0f - 1.0f, uvy = (fy / resy) * 2.0f - 1.0f;  // `uv` varying (camera.vs)
  float seed = rb_cam[s] + fx * resy + fy;  // :38
  const v3 P = mk3(f.eye[0], f.eye[1], f.eye[2]), I = mk3(f.dir[0], f.dir[1], f.dir[2]);
  const v3 basisX = mk3(f.basis_x[0], f.basis_x[1], f.basis_x[2]);  // :39, normalize(cross(I, vec3(0, 1, 0)))
  const v3 basisY = mk3(f.basis_y[0], f.basis_y[1], f.basis_y[2]);  // :40, normalize(cross(basisX, I))
  const float inCamX = uvx * (resx / resy), inCamY = uvy * 1.0f;  // getScreen, :21-24
  const v3 screen = add(add(add(mul(mul(inCamX, basisX), f.fov_scale), mul(mul(inCamY, basisY), f.fov_scale)), I), P);
  const float theta = rnd(seed) * 3.14159265f * 2.0f;  // getAA, :26-30
  const float r = sqrtf(rnd(seed)) * 1.414f;
  float st, ct;
  dm::sincosf_(theta, st, ct);
  v3 aa = mul(r, add(div_shared(mul(basisX, ct), resx), div_shared(mul(basisY, st), resy)));  // (one reciprocal per vector)
  aa = mul(aa, f.fov_scale);  // :42
  const float theta2 = rnd(seed) * 3.14159265f * 2.0f;  // getDOF, :32-35
  float st2, ct2;
  dm::sincosf_(theta2, st2, ct2);
  const v3 dofDir = add(mul(ct2, basisX), mul(st2, basisY));
  const v3 dof = mul(mul(dofDir, f.lens1), sqrtf(rnd(seed)));
  o = add(P, dof);  // :44
  d = normalize_shared(sub(add(add(screen, aa), mul(dof, f.lens0)), add(P, dof)));  // :45
}
