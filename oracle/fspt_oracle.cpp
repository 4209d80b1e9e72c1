/*
 * oracle/fspt_oracle.cpp -- TEST INFRASTRUCTURE.  CPU restatement of the FSPT hot path.
 *
 * PARITY PIN: the reference (apbodnar/FSPT) ships no tests, golden vectors or known-answer data, and no browser /
 * Node / GLSL compiler exists in this image.  What this restatement IS checked against is the reference's own shader
 * text: `make -C oracle ref` compiles /root/reference/shader/{camera,tracer,bvh_test,draw}.fs for the CPU behind a GLSL
 * subset (oracle/glsl_cpu/, output oracle/_ref/libfspt_ref.so), and tests/test_reference_pin.py demands bit-identical
 * camera rays, (index, t, count) records, accumulation targets over several ticks and RGBA8 frames from the two, on
 * four scenes; the fixtures under tests/golden hold outputs of those shaders.  What remains a model on BOTH sides is what GLSL
 * leaves to the platform -- built-in function precision (oracle_math.h, "FSPT-DM2") and texture filtering arithmetic
 * (oracle_texunit.h) -- and the two deliberate guards listed in DESIGN.md section 2 (refraction cap, NaN sanitising,
 * both switchable off and off in those tests).
 *
 * Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference
 * legs may load this library.  The product (fspt_b200/) never does.
 *
 * Every function cites the reference file:line it follows (paths relative to the
 * reference root).  Arithmetic model: oracle_math.h ("FSPT-DM2").
 * Build: g++ -O2 -ffp-contract=off -fno-fast-math (see oracle/Makefile).
 */
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <atomic>
#include <thread>
#include <vector>

#include "oracle_math.h"
#include "oracle_texunit.h"

using namespace om;

extern "C" {

/* The GL resources main.js hands to the tracer program (main.js:360-445,548-560,170-204),
 * un-padded (padBuffer's -1 fill, main.js:143-154, is re-created by the fetch helpers). */
struct OScene {
  const float* bvh;      /* 9 f32 / node, [0..2] = int32 bits (maskBVHBuffer, main.js:272-282) */
  const float* tris;     /* 9 f32 / triangle  (main.js:374)      */
  const float* mats;     /* 12 f32 / triangle (main.js:377-382)  */
  const float* norms;    /* 27 f32 / triangle (main.js:383-385)  */
  const float* uvs;      /* 6 f32 / triangle  (main.js:386)      */
  const uint8_t* atlas;  /* res*res*4*layers  (main.js:556-559)  */
  const uint8_t* env;    /* RGBE-in-RGBA8, row 0 = image top (main.js:170-180) */
  const uint16_t* bins;  /* 4 u16 / bin (env_sampler.js:73)      */
  int32_t n_nodes, n_tris, atlas_res, atlas_layers, env_w, env_h, n_bins, leaf_size;
};

struct OStats {
  uint64_t rays;        /* intersectScene calls                       */
  uint64_t node_visits; /* loop iterations V (tracer.fs:373)          */
  uint64_t leaf_visits; /* processLeaf calls L (tracer.fs:380)        */
  uint64_t stack_overflow;
  uint64_t capped;      /* paths stopped by the refraction safety cap      */
};

}  // extern "C"

namespace {

const int NUM_BOUNCES = 4;            /* tracer.fs:9  */
const float MAX_T = 100000.0f;        /* tracer.fs:10 */
const float EPSILON = 0.000001f;      /* tracer.fs:11 */
const float M_PI_F = 3.14159265f;     /* tracer.fs:12 */
const float M_TAU = M_PI_F * 2.0f;    /* tracer.fs:13 */
const float INV_PI = 1.0f / M_PI_F;   /* tracer.fs:14 */

struct Hit { float t; int index; };
struct Counters { uint64_t rays = 0, nodes = 0, leaves = 0, overflow = 0, capped = 0; };

inline int32_t f2i(float f) { int32_t i; memcpy(&i, &f, 4); return i; }

/* createTriangle, tracer.fs:119-126; out-of-range = padBuffer's (-1,-1,-1) texels */
inline void fetchTriangle(const OScene& s, int index, v3& v1, v3& v2, v3& v3_) {
  if (index < 0 || index >= s.n_tris) {
    v1 = v2 = v3_ = mk3(-1.0f, -1.0f, -1.0f);
    return;
  }
  const float* p = s.tris + (size_t)index * 9;
  v1 = mk3(p[0], p[1], p[2]);
  v2 = mk3(p[3], p[4], p[5]);
  v3_ = mk3(p[6], p[7], p[8]);
}

/* rayTriangleIntersect, tracer.fs:300-315 (== bvh_test.fs:133-148) */
inline float rayTriangleIntersect(v3 ro, v3 rd, v3 tv1, v3 tv2, v3 tv3) {
  v3 e1 = sub(tv2, tv1);
  v3 e2 = sub(tv3, tv1);
  v3 p = cross(rd, e2);
  float det = dot(e1, p);
  if (fabsf(det) < EPSILON) return MAX_T;
  float invDet = 1.0f / det;
  v3 t = sub(ro, tv1);
  float u = dot(t, p) * invDet;
  if (u < 0.0f || u > 1.0f) return MAX_T;
  v3 q = cross(t, e1);
  float v = dot(rd, q) * invDet;
  if (v < 0.0f || u + v > 1.0f) return MAX_T;
  float dist = dot(e2, q) * invDet;
  return dist > EPSILON ? dist : MAX_T;
}

/* rayBoxIntersect, tracer.fs:317-326; box = texels 1,2 of node `index` (tracer.fs:161-169) */
inline float rayBoxIntersect(const OScene& s, int index, v3 ro, v3 rd) {
  const float* n = s.bvh + (size_t)index * 9;
  v3 bMin = mk3(n[3], n[4], n[5]), bMax = mk3(n[6], n[7], n[8]);
  v3 inverse = mk3(1.0f / rd.x, 1.0f / rd.y, 1.0f / rd.z);
  v3 t1 = mul(sub(bMin, ro), inverse);
  v3 t2 = mul(sub(bMax, ro), inverse);
  v3 minT = mk3(fminN(t1.x, t2.x), fminN(t1.y, t2.y), fminN(t1.z, t2.z));
  v3 maxT = mk3(fmaxN(t1.x, t2.x), fmaxN(t1.y, t2.y), fmaxN(t1.z, t2.z));
  float tMax = fminN(fminN(maxT.x, maxT.y), maxT.z);
  float tMin = fmaxN(fmaxN(minT.x, minT.y), minT.z);
  return (tMax >= tMin && tMax > 0.0f) ? tMin : MAX_T;
}

/* intersectScene with the visit counter: bvh_test.fs:173-221 (== tracer.fs:366-404).
 * anyhit: the product's hit-or-miss traversal (FSPT_PARAM_ANYHIT), which finishes the leaf of the first hit and stops
 * there; the reference has no such exit. */
Hit intersectScene(const OScene& s, v3 ro, v3 rd, Counters& c, int* countOut, bool anyhit = false) {
  int stack[256]; /* reference: int stack[64] (tracer.fs:368); overflow is flagged */
  int ptr = 0;
  stack[ptr++] = -1;
  Hit result = {MAX_T, -1};
  int idx = 0;
  int count = 0;
  c.rays++;
  while (idx > -1) {
    count++;
    const float* node = s.bvh + (size_t)idx * 9; /* createNode, tracer.fs:171-179 */
    int leftIndex = f2i(node[0]);
    int rightIndex = f2i(node[1]);
    int triangles = f2i(node[2]);
    float leftHit = rayBoxIntersect(s, leftIndex, ro, rd);
    float rightHit = rayBoxIntersect(s, rightIndex, ro, rd);
    if (triangles > -1) {
      /* processLeaf, tracer.fs:355-364: exactly LEAF_SIZE consecutive triangles */
      c.leaves++;
      for (int i = 0; i < s.leaf_size; ++i) {
        v3 a, b, d;
        fetchTriangle(s, triangles + i, a, b, d);
        float res = rayTriangleIntersect(ro, rd, a, b, d);
        if (res < result.t) {
          result.index = triangles + i;
          result.t = res;
        }
      }
      if (anyhit && result.index != -1) break;
    } else {
      if (leftHit < result.t && rightHit < result.t) {
        int deferred;
        if (leftHit > rightHit) {
          idx = rightIndex;
          deferred = leftIndex;
        } else {
          idx = leftIndex;
          deferred = rightIndex;
        }
        if (ptr >= 64) c.overflow++;
        if (ptr < 256) stack[ptr++] = deferred; else { ptr++; }
        continue;
      } else if (leftHit < result.t) {
        idx = leftIndex;
        continue;
      } else if (rightHit < result.t) {
        idx = rightIndex;
        continue;
      }
    }
    --ptr;
    idx = ptr < 256 ? stack[ptr] : -1;
  }
  c.nodes += (uint64_t)count;
  if (countOut) *countOut = count;
  return result;
}

/* ---- texture units: the GL sampling model lives in oracle_texunit.h (shared with oracle/glsl_cpu) ---- */
inline long long coordToInt(float f) { return tu_coord_to_int(f); }
inline v4 textureAtlas(const OScene& s, float u, float v, float layerf) {
  return tu_texture_array(s.atlas, s.atlas_res, s.atlas_layers, u, v, layerf);
}
inline v4 textureEnv(const OScene& s, float u, float v) { return tu_texture_env(s.env, s.env_w, s.env_h, u, v); }

/* envColor, tracer.fs:410-414: RGBE decode AFTER filtering the encoded texel */
v3 envColor(const OScene& s, float cx, float cy) {
  v4 rgbe = textureEnv(s, cx, cy);
  float p = dm_pow(2.0f, rgbe.w * 255.0f - 128.0f);
  return mk3(rgbe.x * p, rgbe.y * p, rgbe.z * p);
}
/* envSample, tracer.fs:416-419 */
v3 envSample(const OScene& s, v3 dir, float envTheta) {
  float cx = envTheta + dm_atan2(dir.z, dir.x) / M_TAU;
  float cy = dm_asin(-dir.y) * INV_PI + 0.5f;
  return envColor(s, cx, cy);
}

/* ---- per-fragment state of tracer.fs ------------------------------------- */
struct Frag {
  const OScene& s;
  float seed;
  float randBase, envTheta;
  Counters c;
  explicit Frag(const OScene& sc) : s(sc), seed(0), randBase(0), envTheta(0) {}

  /* rnd, tracer.fs:181 */
  float rnd() {
    seed += 0.211324865405187f;
    return fractf(dm_sin(seed) * 43758.5453123f);
  }
  /* sampleEnv, tracer.fs:421-434 */
  v4 sampleEnv() {
    int idx = (int)coordToInt((float)s.n_bins * rnd());
    if (idx >= s.n_bins) idx = s.n_bins - 1; /* fract() may return 1.0; GLSL: OOB uniform read */
    if (idx < 0) idx = 0;
    const uint16_t* bq = s.bins + (size_t)idx * 4;
    float bx = (float)bq[0], by = (float)bq[1], bz = (float)bq[2], bw = (float)bq[3];
    float dimsx = (float)s.env_w, dimsy = (float)s.env_h;
    float r1 = rnd();
    float r2 = rnd();
    float uvx = -envTheta + ((bz - bx) * r1 + bx) / dimsx;
    float uvy = 0.0f + ((bw - by) * r2 + by) / dimsy;
    float theta = uvx * M_TAU;
    float phi = uvy * M_PI_F;
    float sinPhi = dm_sin(phi);
    v4 dirPdf;
    dirPdf.x = dm_cos(theta) * sinPhi;
    dirPdf.y = dm_cos(phi);
    dirPdf.z = dm_sin(theta) * sinPhi;
    float nominal = (dimsx * dimsy) / (float)s.n_bins;
    dirPdf.w = nominal / ((bz - bx) * (bw - by) * M_TAU * M_PI_F * sinPhi);
    return dirPdf;
  }
  /* sampleMicrofacet, tracer.fs:256-270 */
  v3 sampleMicrofacet(v3 normal, v2 mr) {
    float r1 = rnd();
    float r2 = rnd();
    v3 up = fabsf(normal.z) < 0.999f ? mk3(0, 0, 1) : mk3(1, 0, 0);
    v3 tangent = normalize(cross(up, normal));
    v3 bitangent = cross(normal, tangent);
    float a = fmaxN(0.001f, mr.y);
    float phi = r1 * M_TAU;
    float cosTheta = sqrtf((1.0f - r2) / (1.0f + (a * a - 1.0f) * r2));
    float sinTheta = clampf(sqrtf(1.0f - (cosTheta * cosTheta)), 0.0f, 1.0f);
    float sinPhi = dm_sin(phi);
    float cosPhi = dm_cos(phi);
    v3 h = mk3(sinTheta * cosPhi, sinTheta * sinPhi, cosTheta);
    return add(add(mul(tangent, h.x), mul(bitangent, h.y)), mul(normal, h.z));
  }
  /* cosineSampleHemisphere + sampleLambert, tracer.fs:205-213,272-280 */
  v3 sampleLambert(v3 normal) {
    float r1 = rnd();
    float r2 = rnd();
    v3 up = fabsf(normal.z) < 0.999f ? mk3(0, 0, 1) : mk3(1, 0, 0);
    v3 tangent = normalize(cross(up, normal));
    v3 bitangent = cross(normal, tangent);
    v3 dir;
    float r = sqrtf(r1);
    float phi = M_TAU * r2;
    dir.x = r * dm_cos(phi);
    dir.y = r * dm_sin(phi);
    dir.z = sqrtf(fmaxN(0.0f, 1.0f - dir.x * dir.x - dir.y * dir.y));
    return add(add(mul(tangent, dir.x), mul(bitangent, dir.y)), mul(normal, dir.z));
  }
};

/* misWeights, tracer.fs:194-203 */
inline v2 misWeights(float a, float b) {
  v2 r;
  if (a > EPSILON && b > EPSILON) {
    float a2 = a * a, b2 = b * b, a2b2 = a2 + b2;
    r.x = a2 / a2b2;
    r.y = b2 / a2b2;
  } else {
    r.x = 1.0f;
    r.y = 0.0f;
  }
  return r;
}
/* gtr2, smithG: tracer.fs:215-225 */
inline float gtr2(float ndh, float a) {
  float a2 = a * a;
  float t = 1.0f + (a2 - 1.0f) * ndh * ndh;
  return a2 / (M_PI_F * t * t);
}
inline float smithG(float NDotv, float alphaG) {
  float a = alphaG * alphaG;
  float b = NDotv * NDotv;
  return 1.0f / (NDotv + sqrtf(a + b - a * b));
}
/* gtr2Pdf, tracer.fs:227-233 */
inline float gtr2Pdf(v3 incident, v3 normal, v2 mr, v3 bsdfDir) {
  float specularAlpha = fmaxN(0.001f, mr.y);
  v3 halfVec = normalize(add(bsdfDir, incident));
  float cosTheta = fabsf(dot(halfVec, normal));
  float pdfgtr2 = gtr2(cosTheta, specularAlpha) * cosTheta;
  return pdfgtr2 / (4.0f * fabsf(dot(bsdfDir, halfVec)));
}
/* lambertPdf, tracer.fs:235-237 */
inline float lambertPdf(v3 normal, v3 bsdfDir) { return fabsf(dot(bsdfDir, normal)) * INV_PI; }
/* schlick, tracer.fs:239-254 */
inline float schlick(v3 incident, v3 normal, v2 ns) {
  float r0 = (ns.x - ns.y) / (ns.x + ns.y);
  r0 *= r0;
  float cosTheta = dot(normal, incident);
  if (ns.x > ns.y) {
    float n = ns.x / ns.y;
    float sinTheta2 = n * n * (1.0f - cosTheta * cosTheta);
    if (sinTheta2 > 1.0f) return 1.0f;
    cosTheta = sqrtf(1.0f - sinTheta2);
  }
  float x = 1.0f - cosTheta;
  return r0 + (1.0f - r0) * x * x * x * x * x;
}
/* evalSpecular, tracer.fs:282-294 */
inline v3 evalSpecular(v3 incident, v3 normal, v3 diffuseColor, v2 mr, v3 bsdfDir) {
  float ndl = dot(normal, bsdfDir);
  float ndv = dot(normal, incident);
  v3 H = normalize(add(bsdfDir, incident));
  float ndh = dot(normal, H);
  float a = fmaxN(0.001f, mr.y);
  float Ds = gtr2(ndh, a);
  v3 Fs = mix3(mk3(1.0f, 1.0f, 1.0f), diffuseColor, mr.x);
  float roughg = (mr.y * 0.5f + 0.5f);
  roughg = roughg * roughg;
  float Gs = smithG(ndl, roughg) * smithG(ndv, roughg);
  return mul(mul(Gs, Fs), Ds);
}
/* evalLambert, tracer.fs:296-298 */
inline v3 evalLambert(v3 diffuseColor) { return mul(diffuseColor, INV_PI); }

/* barycentricWeights, tracer.fs:339-353 */
inline v3 barycentricWeights(v3 tv1, v3 tv2, v3 tv3, v3 p) {
  v3 v0 = sub(tv2, tv1), v1 = sub(tv3, tv1), v2_ = sub(p, tv1);
  float d00 = dot(v0, v0), d01 = dot(v0, v1), d11 = dot(v1, v1), d20 = dot(v2_, v0), d21 = dot(v2_, v1);
  float invDenom = 1.0f / (d00 * d11 - d01 * d01);
  float v = (d11 * d20 - d01 * d21) * invDenom;
  float w = (d00 * d21 - d01 * d20) * invDenom;
  float u = 1.0f - v - w;
  return mk3(u, v, w);
}

/* tracer.fs main(), :436-518.  Returns the un-clamped path colour. */
v3 tracePixel(Frag& F, v3 rayOrigin, v3 rayDir, int maxRefractions) {
  const OScene& s = F.s;
  /* :438 seed = randBase + gl_FragCoord.x + gl_FragCoord.y*dims.x is overwritten at :458
   * before the first rnd() of every path, so it is not modelled. */
  Hit result = intersectScene(s, rayOrigin, rayDir, F.c, nullptr); /* :440 */
  v3 color = mk3(0, 0, 0);
  if (result.index < 0) {
    color = add(color, envSample(s, rayDir, F.envTheta)); /* :443 */
  } else {
    v3 accumulatedReflectance = mk3(1, 1, 1);
    int refractions = 0;
    for (int i = 0; i < NUM_BOUNCES; ++i) {
      /* createMaterial/createTriangle/createTexCoords, :447-449 */
      const float* m = s.mats + (size_t)result.index * 12;
      float mapDiffuse = m[0], mapSpecular = m[1], mapNormal = m[2], mapRoughness = m[3];
      float matIor = m[9], matDielectric = m[10];
      v3 tv1, tv2, tv3;
      fetchTriangle(s, result.index, tv1, tv2, tv3);
      const float* uvp = s.uvs + (size_t)result.index * 6;
      v3 origin = add(rayOrigin, mul(rayDir, result.t));            /* :450 */
      v3 bw = barycentricWeights(tv1, tv2, tv3, origin);            /* :451 */
      float tcx = bw.x * uvp[0] + bw.y * uvp[2] + bw.z * uvp[4];    /* :452, :328-330 */
      float tcy = bw.x * uvp[1] + bw.y * uvp[3] + bw.z * uvp[5];
      v4 tD = textureAtlas(s, tcx, tcy, mapDiffuse);                /* :453 */
      v4 tE = textureAtlas(s, tcx, tcy, mapSpecular);               /* :454 */
      v4 tMR = textureAtlas(s, tcx, tcy, mapRoughness);             /* :455 */
      v4 tN = textureAtlas(s, tcx, tcy, mapNormal);                 /* :456 */
      v3 texDiffuse = mk3(tD.x, tD.y, tD.z);
      v3 texEmmissive = mk3(tE.x, tE.y, tE.z);
      v2 texMR = {tMR.x, tMR.y};
      v3 texNormal = mul(sub(mk3(tN.x, tN.y, tN.z), mk3(0.5f, 0.5f, 0.0f)), mk3(2.0f, 2.0f, 1.0f));
      texMR.y *= texMR.y;                                           /* :457 */
      F.seed = origin.x * F.randBase * origin.y * 1.396529836f + origin.z * 4761.52835f; /* :458 */
      /* createNormals + barycentricNormal, :137-150, :332-337, :460 */
      const float* np = s.norms + (size_t)result.index * 27;
      v3 n1 = mk3(np[0], np[1], np[2]), t1 = mk3(np[3], np[4], np[5]), b1 = mk3(np[6], np[7], np[8]);
      v3 n2 = mk3(np[9], np[10], np[11]), t2 = mk3(np[12], np[13], np[14]), b2 = mk3(np[15], np[16], np[17]);
      v3 n3 = mk3(np[18], np[19], np[20]), t3 = mk3(np[21], np[22], np[23]), b3 = mk3(np[24], np[25], np[26]);
      v3 baryNormal = add(add(mul(bw.x, n1), mul(bw.y, n2)), mul(bw.z, n3));
      v3 baryTangent = add(add(mul(bw.x, t1), mul(bw.y, t2)), mul(bw.z, t3));
      v3 baryBiTangent = add(add(mul(bw.x, b1), mul(bw.y, b2)), mul(bw.z, b3));
      v3 macroNormal = normalize(add(add(mul(texNormal.x, baryTangent), mul(texNormal.y, baryBiTangent)),
                                     mul(texNormal.z, baryNormal)));
      bool inside = dot(neg(rayDir), baryNormal) < 0.0f;            /* :461 */
      v2 ns;
      if (inside) { ns.x = matIor; ns.y = 1.0f; } else { ns.x = 1.0f; ns.y = matIor; } /* :462 */
      macroNormal = inside ? neg(macroNormal) : macroNormal;        /* :463 */
      rayOrigin = add(origin, mul(mul(macroNormal, EPSILON), 2.0f)); /* :464 */

      color = add(color, mul(mul(mul(accumulatedReflectance, texEmmissive), texDiffuse), 30.0f)); /* :467 */
      v3 incident = neg(rayDir);
      v3 envThroughput, bsdfThroughput;
      float bsdfPdf;
      v3 microNormal = F.sampleMicrofacet(macroNormal, texMR);      /* :472 */
      v4 envDirPdf = F.sampleEnv();                                 /* :473 */
      v3 envDir = mk3(envDirPdf.x, envDirPdf.y, envDirPdf.z);
      float cosEnv = dot(macroNormal, envDir);                      /* :474 */
      bool specular = mixf(schlick(incident, microNormal, ns), 1.0f, texMR.x) > F.rnd(); /* :475 */
      if (specular) {
        rayDir = reflect(neg(incident), microNormal);               /* :477 */
        bsdfPdf = gtr2Pdf(incident, macroNormal, texMR, rayDir);    /* :478 */
        bsdfThroughput = div(mul(evalSpecular(incident, macroNormal, texDiffuse, texMR, rayDir),
                                 clampf(dot(macroNormal, rayDir), 0.0f, 1.0f)), bsdfPdf); /* :479 */
        envThroughput = div(mul(evalSpecular(incident, macroNormal, texDiffuse, texMR, envDir),
                                clampf(cosEnv, 0.0f, 1.0f)), envDirPdf.w);                /* :480 */
      } else if (matDielectric >= 0.0f) {
        bsdfPdf = 1.0f;
        bsdfThroughput = mk3(1, 1, 1);
        envThroughput = mk3(0, 0, 0);
        rayOrigin = sub(origin, mul(mul(macroNormal, EPSILON), 2.0f)); /* :485 */
        rayDir = refract(neg(incident), microNormal, ns.x / ns.y);     /* :486 */
        i--;                                                           /* :488 */
        /* the reference loop is unbounded here; cap documented in DESIGN.md */
        if (++refractions > maxRefractions) { i = NUM_BOUNCES; F.c.capped++; }
      } else {
        rayDir = F.sampleLambert(macroNormal);                      /* :490 */
        bsdfPdf = lambertPdf(macroNormal, rayDir);                  /* :491 */
        bsdfThroughput = div(mul(evalLambert(texDiffuse), clampf(dot(macroNormal, rayDir), 0.0f, 1.0f)), bsdfPdf);
        envThroughput = div(mul(evalLambert(texDiffuse), clampf(cosEnv, 0.0f, 1.0f)), envDirPdf.w);
      }
      /* Beer's-law override, :497 */
      if (inside) {
        v3 om_ = sub(mk3(1, 1, 1), texDiffuse);
        v3 b = sub(mk3(1, 1, 1), mul(mul(om_, result.t), matDielectric));
        bsdfThroughput = mk3(fmaxN(b.x, 0.0f), fmaxN(b.y, 0.0f), fmaxN(b.z, 0.0f));
      }
      v2 weights = misWeights(envDirPdf.w, bsdfPdf);                /* :499 */
      if (matDielectric < 0.0f && cosEnv > 0.0f) {                  /* :500 */
        Hit shadow = intersectScene(s, rayOrigin, envDir, F.c, nullptr);
        if (shadow.index == -1) {
          color = add(color, mul(mul(mul(accumulatedReflectance, envThroughput), envSample(s, envDir, F.envTheta)),
                                 weights.x));                       /* :503 */
        }
      }
      result = intersectScene(s, rayOrigin, rayDir, F.c, nullptr);  /* :507 */
      accumulatedReflectance = mul(accumulatedReflectance, bsdfThroughput); /* :508 */
      if (result.index == -1) {
        color = add(color, mul(mul(accumulatedReflectance, envSample(s, rayDir, F.envTheta)), weights.y)); /* :510 */
        break;
      }
    }
  }
  return color;
}

template <class Fn>
void parallelRows(int rows, int nthreads, Fn fn) {
  if (nthreads <= 0) nthreads = (int)std::thread::hardware_concurrency();
  if (nthreads < 1) nthreads = 1;
  if (nthreads > rows) nthreads = rows > 0 ? rows : 1;
  std::atomic<int> next(0);
  std::vector<std::thread> th;
  for (int t = 0; t < nthreads; ++t)
    th.emplace_back([&, t]() {
      for (;;) {
        int r = next.fetch_add(1);
        if (r >= rows) break;
        fn(r, t);
      }
    });
  for (auto& x : th) x.join();
}

}  // namespace

extern "C" {

int oracle_abi_version() { return 1; }

/* ---- det-math probes (so tests can pin FSPT-DM2 against libm and the GPU) ----
 * The codes are fspt_debug_math's (include/fspt_b200.h); each answers with the model's plain operation: the device's
 * division shortcuts (13-15) all answer x / y, sincos (6, 7) answers sin / cos, the packed slab-test lanes (32-35) the
 * scalar subtraction / multiplication of their operands.  Returns -1 for an unknown code. */
int oracle_dm_eval(int fn, const float* x, const float* y, float* out, int n) {
  if (fn < 0 || (fn > 17 && (fn < 32 || fn > 35))) return -1;
  for (int i = 0; i < n; ++i) {
    switch (fn) {
      case 0: case 6: out[i] = dm_sin(x[i]); break;
      case 1: case 7: out[i] = dm_cos(x[i]); break;
      case 2: out[i] = dm_atan2(y[i], x[i]); break;
      case 3: out[i] = dm_asin(x[i]); break;
      case 4: out[i] = dm_exp2(x[i]); break;
      case 5: out[i] = dm_pow(x[i], y[i]); break;
      case 8: out[i] = dm_log2(x[i]); break;
      case 9: out[i] = fractf(dm_sin(x[i]) * 43758.5453123f); break;
      case 10: out[i] = fminN(x[i], y[i]); break;
      case 11: out[i] = fmaxN(x[i], y[i]); break;
      case 12: out[i] = clampf(x[i], 0.0f, 1024.0f); break;
      case 13: case 14: case 15: out[i] = x[i] / y[i]; break;
      case 16: { const int32_t v = (int32_t)tu_coord_to_int(x[i]); memcpy(&out[i], &v, 4); break; }
      case 17: out[i] = (float)tu_quant8(x[i]); break;
      case 32: out[i] = x[i] - y[i]; break;
      case 33: out[i] = -x[i] - y[i]; break;
      case 34: out[i] = x[i] * y[i]; break;
      case 35: out[i] = -x[i] * y[i]; break;
    }
  }
  return 0;
}

/* camera.fs main(), :37-46.  Outputs RGBA32F pos/dir, index = y*W + x, y up (gl_FragCoord). */
void oracle_camera(int W, int H, const float* P, const float* I, float fovScale, const float* lens,
                   float randBase, float* pos4, float* dir4, int nthreads) {
  v3 Pv = mk3(P[0], P[1], P[2]), Iv = mk3(I[0], I[1], I[2]);
  float resx = (float)W, resy = (float)H;
  const float M_PI_C = 3.14159265f; /* camera.fs:11 */
  parallelRows(H, nthreads, [&](int y, int) {
    for (int x = 0; x < W; ++x) {
      float fx = (float)x + 0.5f, fy = (float)y + 0.5f; /* gl_FragCoord */
      /* `uv` varying = corner.xy interpolated over the oversized triangle (camera.vs, main.js:601-605) */
      float uvx = (fx / resx) * 2.0f - 1.0f, uvy = (fy / resy) * 2.0f - 1.0f;
      float seed = randBase + fx * resy + fy; /* :38 */
      auto rnd = [&]() { seed += 0.211324865405187f; return fractf(dm_sin(seed) * 43758.5453123f); }; /* :19 */
      v3 basisX = normalize(cross(Iv, mk3(0, 1, 0)));  /* :39 */
      v3 basisY = normalize(cross(basisX, Iv));        /* :40 */
      /* getScreen, :21-24 */
      float inCamX = uvx * (resx / resy), inCamY = uvy * 1.0f;
      v3 screen = add(add(add(mul(mul(inCamX, basisX), fovScale), mul(mul(inCamY, basisY), fovScale)), Iv), Pv);
      /* getAA, :26-30 */
      float theta = rnd() * M_PI_C * 2.0f;
      float r = sqrtf(rnd()) * 1.414f;
      v3 aa = mul(r, add(div(mul(basisX, dm_cos(theta)), resx), div(mul(basisY, dm_sin(theta)), resy)));
      aa = mul(aa, fovScale); /* :42 */
      /* getDOF, :32-35 */
      float theta2 = rnd() * M_PI_C * 2.0f;
      v3 dofDir = add(mul(dm_cos(theta2), basisX), mul(dm_sin(theta2), basisY));
      v3 dof = mul(mul(dofDir, lens[1]), sqrtf(rnd()));
      v3 o = add(Pv, dof); /* :44 */
      v3 d = normalize(sub(add(add(screen, aa), mul(dof, lens[0])), add(Pv, dof))); /* :45 */
      size_t k = ((size_t)y * W + x) * 4;
      pos4[k] = o.x; pos4[k + 1] = o.y; pos4[k + 2] = o.z; pos4[k + 3] = 1.0f;
      dir4[k] = d.x; dir4[k + 1] = d.y; dir4[k + 2] = d.z; dir4[k + 3] = 1.0f;
    }
  });
}

/* bvh_test.fs main(), :224-232, exporting (result.index, result.t, count) instead of the heat-map; anyhit != 0 traces
 * every ray hit-or-miss (see intersectScene) */
void oracle_bvh_test(const OScene* s, const float* pos4, const float* dir4, int n, int32_t* index, float* t,
                     int32_t* count, OStats* stats, int nthreads, int anyhit) {
  int chunk = 4096;
  int rows = (n + chunk - 1) / chunk;
  std::vector<Counters> cs(256);
  if (nthreads <= 0) nthreads = (int)std::thread::hardware_concurrency();
  if (nthreads > 256) nthreads = 256;
  parallelRows(rows, nthreads, [&](int r, int tid) {
    int lo = r * chunk, hi = std::min(n, lo + chunk);
    for (int i = lo; i < hi; ++i) {
      v3 o = mk3(pos4[4 * (size_t)i], pos4[4 * (size_t)i + 1], pos4[4 * (size_t)i + 2]);
      v3 d = mk3(dir4[4 * (size_t)i], dir4[4 * (size_t)i + 1], dir4[4 * (size_t)i + 2]);
      int cnt = 0;
      Hit h = intersectScene(*s, o, d, cs[tid], &cnt, anyhit != 0);
      index[i] = h.index;
      t[i] = h.t;
      count[i] = cnt;
    }
  });
  if (stats) {
    for (auto& c : cs) {
      stats->rays += c.rays; stats->node_visits += c.nodes; stats->leaf_visits += c.leaves;
      stats->stack_overflow += c.overflow;
    }
  }
}

/* brute force over all triangles with the same Moller-Trumbore arithmetic (test aid) */
void oracle_brute_force(const OScene* s, const float* pos4, const float* dir4, int n, int32_t* index, float* t,
                        int nthreads) {
  int chunk = 256;
  int rows = (n + chunk - 1) / chunk;
  parallelRows(rows, nthreads, [&](int r, int) {
    int lo = r * chunk, hi = std::min(n, lo + chunk);
    for (int i = lo; i < hi; ++i) {
      v3 o = mk3(pos4[4 * (size_t)i], pos4[4 * (size_t)i + 1], pos4[4 * (size_t)i + 2]);
      v3 d = mk3(dir4[4 * (size_t)i], dir4[4 * (size_t)i + 1], dir4[4 * (size_t)i + 2]);
      Hit h = {MAX_T, -1};
      for (int k = 0; k < s->n_tris; ++k) {
        v3 a, b, c;
        fetchTriangle(*s, k, a, b, c);
        float res = rayTriangleIntersect(o, d, a, b, c);
        if (res < h.t) { h.t = res; h.index = k; }
      }
      index[i] = h.index;
      t[i] = h.t;
    }
  });
}

/* One drawTracer() pass (main.js:758-807 + tracer.fs main): fb_out = (color + fb_prev*tick)/(tick+1).
 * fb_* are RGBA32F, y up.  color_out (optional) receives the clamped per-sample colour. */
void oracle_trace(const OScene* s, const float* pos4, const float* dir4, int W, int H, uint32_t tick,
                  float randBase, float envTheta, const float* fb_prev, float* fb_out, float* color_out,
                  int sanitize, int maxRefractions, OStats* stats, int nthreads) {
  if (nthreads <= 0) nthreads = (int)std::thread::hardware_concurrency();
  if (nthreads > 256) nthreads = 256;
  std::vector<Counters> cs(256);
  parallelRows(H, nthreads, [&](int y, int tid) {
    Frag F(*s);
    F.randBase = randBase;
    F.envTheta = envTheta;
    for (int x = 0; x < W; ++x) {
      size_t k = ((size_t)y * W + x) * 4;
      v3 o = mk3(pos4[k], pos4[k + 1], pos4[k + 2]), d = mk3(dir4[k], dir4[k + 1], dir4[k + 2]);
      v3 color = tracePixel(F, o, d, maxRefractions);
      if (sanitize) { /* deviation: the reference lets NaN stick in the accumulator (tracer.fs:515-517) */
        if (color.x != color.x) color.x = 0.0f;
        if (color.y != color.y) color.y = 0.0f;
        if (color.z != color.z) color.z = 0.0f;
      }
      color = clamp3(color, 0.0f, 1024.0f); /* :515 */
      if (color_out) { color_out[k] = color.x; color_out[k + 1] = color.y; color_out[k + 2] = color.z; color_out[k + 3] = 1.0f; }
      v3 tcolor = fb_prev ? mk3(fb_prev[k], fb_prev[k + 1], fb_prev[k + 2]) : mk3(0, 0, 0); /* :516 */
      float ft = (float)tick;
      v3 outc = div(add(color, mul(tcolor, ft)), ft + 1.0f); /* :517 */
      fb_out[k] = outc.x; fb_out[k + 1] = outc.y; fb_out[k + 2] = outc.z; fb_out[k + 3] = 1.0f;
    }
    cs[tid].rays += F.c.rays; cs[tid].nodes += F.c.nodes; cs[tid].leaves += F.c.leaves; cs[tid].overflow += F.c.overflow;
    cs[tid].capped += F.c.capped;
  });
  if (stats)
    for (auto& c : cs) {
      stats->rays += c.rays; stats->node_visits += c.nodes; stats->leaf_visits += c.leaves;
      stats->stack_overflow += c.overflow; stats->capped += c.capped;
    }
}

/* draw.fs main(), :82-93 (+ filterFireflies :50-80, ACESFitted :39-48).  RGBA8 out, y up. */
void oracle_draw(const float* fb, int W, int H, float exposure, float saturation, int denoise, float maxSigma,
                 float scale, uint8_t* rgba8, int nthreads) {
  const v3 lumaCoefs = mk3(0.2126f, 0.7152f, 0.0722f);
  auto fetch = [&](long long cx, long long cy) -> v3 { /* texelFetch; out of range = 0 (robust access) */
    if (cx < 0 || cy < 0 || cx >= W || cy >= H) return mk3(0, 0, 0);
    const float* p = fb + ((size_t)cy * W + (size_t)cx) * 4;
    return mk3(p[0], p[1], p[2]);
  };
  parallelRows(H, nthreads, [&](int y, int) {
    for (int x = 0; x < W; ++x) {
      float fx = (float)x + 0.5f, fy = (float)y + 0.5f;
      long long bx = coordToInt(fx * scale), by = coordToInt(fy * scale); /* ivec2(gl_FragCoord*scale) */
      v3 texColor;
      if (denoise) {
        float sum = 0.0f, sq_sum = 0.0f;
        v3 middle = mk3(0, 0, 0);
        float middleLuma = 0.0f;
        const int KERNEL_SIZE = 5;
        float samples = (float)(KERNEL_SIZE * KERNEL_SIZE) - 1.0f;
        for (int i = 0; i < KERNEL_SIZE; i++)
          for (int j = 0; j < KERNEL_SIZE; j++) {
            int osx = i - KERNEL_SIZE / 2, osy = j - KERNEL_SIZE / 2;
            v3 color = fetch(bx + osx, by + osy);
            float luma = dot(color, lumaCoefs);
            if (osx == 0 && osy == 0) { middle = color; middleLuma = luma; continue; }
            sum += luma;
            sq_sum += luma * luma;
          }
        float mean = sum / samples;
        float variance = sq_sum / samples - mean * mean;
        float sigma = sqrtf(variance);
        if (fabsf(middleLuma - mean) > maxSigma * sigma) middle = mul(middle, mean / middleLuma);
        texColor = mul(middle, exposure);
      } else {
        texColor = mul(fetch(bx, by), exposure);
      }
      /* ACESFitted: color * ACESInputMat (row vector x column-major mat3), draw.fs:19-48 */
      v3 c = texColor;
      v3 a = mk3(c.x * 0.59719f + c.y * 0.35458f + c.z * 0.04823f,
                 c.x * 0.07600f + c.y * 0.90834f + c.z * 0.01566f,
                 c.x * 0.02840f + c.y * 0.13383f + c.z * 0.83777f);
      auto fit = [](float v) {
        float aa = v * (v + 0.0245786f) - 0.000090537f;
        float bb = v * (0.983729f * v + 0.4329510f) + 0.238081f;
        return aa / bb;
      };
      a = mk3(fit(a.x), fit(a.y), fit(a.z));
      v3 o = mk3(a.x * 1.60475f + a.y * -0.53108f + a.z * -0.07367f,
                 a.x * -0.10208f + a.y * 1.10813f + a.z * -0.00605f,
                 a.x * -0.00327f + a.y * -0.07276f + a.z * 1.07602f);
      v3 mapped = clamp3(o, 0.0f, 1.0f);
      float l = dot(mapped, lumaCoefs);
      mapped = mix3(mk3(l, l, l), mapped, saturation);
      mapped = mk3(dm_pow(mapped.x, 0.454545f), dm_pow(mapped.y, 0.454545f), dm_pow(mapped.z, 0.454545f));
      auto q8 = [](float v) -> uint8_t { /* RGBA8 framebuffer write: clamp, round to nearest */
        if (!(v > 0.0f)) return 0;
        if (v >= 1.0f) return 255;
        return (uint8_t)(int)floorf(v * 255.0f + 0.5f);
      };
      uint8_t* out = rgba8 + ((size_t)y * W + x) * 4;
      out[0] = q8(mapped.x); out[1] = q8(mapped.y); out[2] = q8(mapped.z); out[3] = 255;
    }
  });
}

}  // extern "C"
