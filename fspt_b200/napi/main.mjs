// main.mjs -- headless Node.js host: main.js's tick() loop (main.js:838-857) over the N-API addon.
// Not runnable in this image (no Node); the tested host is fspt_b200/path_tracer.py, which makes the same calls.
//
//   node main.mjs scene.flat.json out.rgba 1280 720 64 [maxRelError]
//
// With maxRelError, the render is adaptive (sum mode): batches of 16 samples until no pixel is active or the 64 are spent.
//
// `scene.flat.json` holds the flattened arrays initBVH() builds (main.js:360-445) as base64 typed arrays; a
// reference maintainer would instead call fspt.sceneUpload() at the end of initBVH() with the arrays it already has.
import { createRequire } from 'module';
import fs from 'fs';
const require = createRequire(import.meta.url);
const fspt = require('./build/Release/fspt_napi.node');

function mulberry32(a) {            // seeded stand-in for Math.random (main.js:748,777)
  return () => { a |= 0; a = a + 0x6D2B79F5 | 0; let t = Math.imul(a ^ a >>> 15, 1 | a);
    t = t + Math.imul(t ^ t >>> 7, 61 | t) ^ t; return ((t ^ t >>> 14) >>> 0) / 4294967296; };
}
const b64 = (s, T) => { const b = Buffer.from(s, 'base64'); return new T(b.buffer, b.byteOffset, b.length / T.BYTES_PER_ELEMENT); };

const [, , scenePath, outPath, W = '1280', H = '720', SPP = '64', ERR] = process.argv;
const s = JSON.parse(fs.readFileSync(scenePath, 'utf8'));
const resolution = [parseInt(W), parseInt(H)];
const ctx = fspt.create(resolution[0], resolution[1], 0);          // initGL + initBuffers
fspt.sceneUpload(ctx, {                                            // the texImage2D/3D uploads of initBVH/initAtlas
  bvh: b64(s.bvh, Float32Array), triangles: b64(s.triangles, Float32Array), materials: b64(s.materials, Float32Array),
  normals: b64(s.normals, Float32Array), uvs: b64(s.uvs, Float32Array), atlas: b64(s.atlas, Uint8Array),
  env: b64(s.env, Uint8Array), radianceBins: b64(s.radianceBins, Uint16Array),
  atlasRes: s.atlasRes, atlasLayers: s.atlasLayers, envWidth: s.envWidth, envHeight: s.envHeight, leafSize: 4,
});
const frame = { eye: s.cameraPos || [0, 0, 2], dir: s.cameraDir || [0, 0, -1], fovScale: s.fovScale || 0.5,
  lensFeatures: [1 - 1 / (s.focalDepth || 2.0), s.aperture ?? 0.02], envTheta: s.environmentTheta || 0 };
const max = parseInt(SPP), rnd = mulberry32(1);
const rc = new Float32Array(max), rt = new Float32Array(max);
for (let i = 0; i < max; i++) { rc[i] = rnd() * 10000; rt[i] = rnd() * 10000; }   // drawCamera, drawTracer
fspt.clear(ctx);
if (ERR === undefined) {
  fspt.render(ctx, frame, 0, rc, rt);                              // max x { drawCamera(); drawTracer(pingpong++) }
} else {                                                           // adaptive: stop the pixels whose mean has converged
  fspt.setAccumMode(ctx, 1);
  fspt.setAdaptive(ctx, parseFloat(ERR), 16);
  for (let t = 0; t < max && fspt.activePixels(ctx) > 0; t += 16) {
    const n = Math.min(16, max - t);
    fspt.render(ctx, frame, t, rc.subarray(t, t + n), rt.subarray(t, t + n));
  }
}
const rgba = fspt.resolve(ctx, { exposure: s.exposure || 1, saturation: 1, maxSigma: 2, scale: 1, denoise: 0 },
  resolution[0], resolution[1]);                                   // drawQuad + readback (GL row order, bottom-up)
fs.writeFileSync(outPath, Buffer.from(rgba.buffer));
