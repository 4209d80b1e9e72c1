"""Host-side mirror of main.js's `PathTracer` closure (main.js:17-951) for a headless host: the same state
(eye, dir, fovScale, lensFeatures, envTheta, exposure, saturation, denoise, maxSigma, pingpong) and the same
entry points (drawCamera+drawTracer = tick, drawQuad, clear, shootAutoFocusRay), driving libfspt_b200.so
through its C ABI instead of WebGL.  The Node.js equivalent over N-API is fspt_b200/napi/ (INTEGRATION.md).
"""
import numpy as np

from . import capi, scenes


class PathTracer:
    def __init__(self, scene_arrays, resolution, camera=None, device=0, seed=1, exposure=1.0, saturation=1.0,
                 denoise=False, max_sigma=2.0, max_samples=2000, async_upload=False):
        self.resolution = (int(resolution[0]), int(resolution[1]))
        cam = dict(eye=[0, 0, 2], dir=[0, 0, -1], fov_scale=0.5, env_theta=0.0, aperture=0.02, focal_depth=2.0)  # main.js:69-74
        cam.update(camera or {})
        self.eye, self.dir = list(cam["eye"]), list(cam["dir"])
        self.fovScale, self.envTheta = cam["fov_scale"], cam["env_theta"]
        self.lensFeatures = scenes.lens_features(cam)
        self.exposure, self.saturation, self.denoise, self.maxSigma = exposure, saturation, denoise, max_sigma
        self.maxSamples = max_samples          # elements.sampleInputElement.value (main.js:67)
        self.pingpong = 0                      # main.js:25
        self.scene = scene_arrays
        self.ctx = capi.Context(self.resolution[0], self.resolution[1], device)
        # scene_arrays None: the scene arrives later (fspt_scene_broadcast from the rank that compiled it)
        # async_upload=True: fspt_scene_upload_async -- the atlas is still being staged when this returns and the first
        # tick's primary traversal overlaps it; self.scene keeps the arrays alive and they must not be modified before then.
        # Default: the synchronous upload, which like texImage2D has consumed every buffer when it returns.
        self.upload_bytes = self.ctx.scene_upload(scene_arrays, wait=not async_upload) if scene_arrays is not None else 0
        self._seed = seed
        self._rand = scenes.rand_bases

    @classmethod
    def from_scene(cls, scene_path, resolution, asset_root=None, device=0, seed=1, autofocus=True, **kw):
        """PathTracer(scenePath, ...) (main.js:915-950 -> start(), :879-913): compile the scene JSON, upload,
        shoot the autofocus ray."""
        from . import scene_json
        sa, cam = scene_json.load_scene(scene_path, asset_root, device=device)
        pt = cls(sa, resolution, cam, device=device, seed=seed, exposure=cam.get("exposure", 1.0),
                 max_samples=cam.get("samples", 2000), **kw)
        if autofocus:
            # the reference shoots the ray through its f64 Triangle.verts, not through the f32 upload (main.js:447-546)
            v64 = sa.verts64 if sa.verts64 is not None else sa.tris.astype(np.float64)
            dist = scene_json.autofocus_distance(v64, pt.eye, pt.dir)
            pt.lensFeatures[0] = 1.0 - 1.0 / dist   # main.js:543-544
        return pt

    # -- main.js:826-836
    def clear(self):
        self.ctx.clear()
        self.pingpong = 0

    def _frame(self):
        return self.ctx.frame(self.eye, self.dir, self.fovScale, self.lensFeatures, self.envTheta)

    # -- main.js:838-857: n iterations of { drawCamera(); drawTracer(pingpong); pingpong++ }
    def tick(self, n=1, rand_base_camera=None, rand_base_tracer=None):
        if rand_base_camera is None:
            # the two Math.random()*10000 draws per iteration (main.js:748,777), from a seeded stream
            rc, rt = self._rand(self.pingpong + n, self._seed)
            rand_base_camera, rand_base_tracer = rc[self.pingpong:], rt[self.pingpong:]
        self.ctx.render(self._frame(), self.pingpong, rand_base_camera, rand_base_tracer)
        self.pingpong += n

    # -- drawQuad (main.js:809-824) + canvas.toBlob (main.js:861): RGBA8, GL row order (row 0 = bottom)
    def drawQuad(self, out=None):
        return self.ctx.resolve(self.exposure, self.saturation, self.denoise, self.maxSigma, 1.0, out)

    def image(self):
        """Top-down RGB image as the canvas shows it."""
        return self.drawQuad()[::-1, :, :3]

    def render(self, samples=None):
        """Run to the sample budget like the rAF loop does (renders max+1 passes: `pingpong <= max`, main.js:841)."""
        samples = self.maxSamples + 1 if samples is None else samples
        if samples > self.pingpong:
            self.tick(samples - self.pingpong)
        return self.drawQuad()

    def converge(self, max_rel_error, max_samples=None, min_samples=16, batch=16):
        """Render until every pixel's mean has converged (adaptive sampling, fspt_set_adaptive) or the sample budget is
        spent (default maxSamples + 1, as in render()), in calls of `batch` ticks; no reference counterpart.  Clears
        first and leaves the context in sum mode with adaptive sampling on, so later tick() calls go on refining the
        pixels that are still active.  Returns drawQuad()."""
        budget = self.maxSamples + 1 if max_samples is None else int(max_samples)
        self.clear()
        self.ctx.set_accum_mode(1)
        self.ctx.set_adaptive(max_rel_error, min_samples)
        while self.pingpong < budget and self.ctx.active_pixels() > 0:
            self.tick(min(batch, budget - self.pingpong))
        return self.drawQuad()

    # -- shootAutoFocusRay (main.js:447-546): one ray along the camera axis -> lensFeatures[0] = 1 - 1/dist.
    # The reference walks its JS tree in float64 with maxT = 1e6; here the same query is one GPU ray (f32,
    # MAX_T = 1e5), which differs from the JS value by f32 rounding of the distance.
    def shootAutoFocusRay(self):
        pos = np.array([[self.eye[0], self.eye[1], self.eye[2], 1.0]], np.float32)
        d = np.array([[self.dir[0], self.dir[1], self.dir[2], 1.0]], np.float32)
        idx, t, _ = self.ctx.debug_trace(pos, d)
        dist = float(t[0]) if idx[0] >= 0 else 1e6
        self.lensFeatures[0] = 1.0 - 1.0 / dist
        return dist

    def accumulation(self):
        return self.ctx.read_accum()

    def stats(self):
        return self.ctx.stats()

    def close(self):
        self.ctx.close()
