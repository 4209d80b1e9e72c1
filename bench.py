#!/usr/bin/env python
"""bench.py -- the reference's headline metric (BASELINE.json): Mpath-samples/s (and Mrays/s) on the bunny-class
scene at 1280x720, 64 spp, bokeh DoF + HDRi importance sampling, on 1/2/4/8 B200.

  python bench.py --gpus N --steps K --warmup W            (N>1: launched by torch.distributed.run)
  python bench.py --impl reference ...                     (the reference's algorithm on the host CPU)
  python bench.py --config {1..5}                          (the other BASELINE.json configs; default 2 = the metric's)
  python bench.py --gpus N --scaling strong                (ONE fixed frame split over N GPUs by tiles x sample sets)
  python bench.py ... --dump-outputs DIR                   (the last timed step's accumulation buffer -> DIR/accum.npy)

A "step" = one frame of the workload (config 2: 64 spp of 1280x720 = 58.98 M path samples).
  value : device-resident throughput -- scene already in HBM, CUDA events on the library's launch stream around
          camera + traversal + shading + accumulation (+ the NCCL reduce for N>1), max over ranks.
  e2e   : the same frame through the public host API with HOST buffers: scene upload (H2D; N>1: rank 0 uploads,
          the other ranks receive it with fspt_scene_broadcast over NVLink) + render + reduce + post-pass + RGBA8
          read-back (D2H) inside the timed region, wall clock bracketed by synchronize + barrier.
  parity: a small frame rendered through the SAME multi-rank path (sharding, collectives behind the C ABI) compared
          bit for bit with the CPU oracle, outside the timed region.
Multi-GPU: every collective runs inside the library (fspt_comm_init / fspt_reduce_accum / fspt_scene_broadcast);
torch.distributed only launches the ranks and carries the NCCL unique id.
  weak   (default, what the driver's scaling run measures): every rank renders its own --spp samples of the frame
         (sample-set sharding), one ncclReduce(sum) per frame.
  strong : the frame's --spp samples are fixed; ranks split it by tiles x sample sets (fspt_b200.dist.partition).
"""
import argparse
import json
import os
import shutil
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "Mpath-samples/s"

# BASELINE.json configs; "spp" is what one bench step renders (config 5: a 64-sample slice of its 1024 spp)
CONFIGS = {
    1: dict(name="configs[0]: bunny-class scene, 800x800, 1 spp (the reference's own CPU-runnable case)",
            scene="bunny", res=(800, 800), spp=1),
    2: dict(name="configs[1]: bunny-class scene, 1280x720, 64 spp, aperture 0.02 DoF, env NEE+MIS", scene="bunny",
            res=(1280, 720), spp=64),
    3: dict(name="configs[2]: 327680-triangle icosphere + 672320-triangle soup (1.0 M), 1280x720, primary + 4 bounces, "
                 "Lambert 0.8", scene="soup", res=(1280, 720), spp=16),
    4: dict(name="configs[3]: textured PBR scene (all four atlas maps, refractive prop ior 1.4), 1920x1080, 256 spp",
            scene="pbr", res=(1920, 1080), spp=256),
    5: dict(name="configs[4]: 10 M-triangle scene (subdiv-8 icosphere + 8.69 M soup, seed 4321), 3840x2160, one "
                 "64-sample slice of the 1024 spp per step", scene="soup10m", res=(3840, 2160), spp=64),
}


def build_scene(args, host=None):
    from fspt_b200 import scenes
    kind = CONFIGS[args.config]["scene"]
    if kind == "bunny":
        return scenes.bunny_class(subdiv=args.subdiv, atlas_res=args.atlas_res, env_size=(2048, 1024), host=host)
    if kind == "soup":
        return scenes.sphere_soup()
    if kind == "pbr":
        return scenes.pbr_scene(atlas_res=args.atlas_res)
    if kind == "soup10m":
        return scenes.sphere_soup(subdiv=8, n_soup=10000000 - 1310720, seed=4321)
    raise ValueError(kind)


def workload_config(args, sa, n_gpus, parallelism):
    cfg = CONFIGS[args.config]
    l2 = ("L2 flushed (512 MB write) between timed steps; per-wave path state (2 x 80 B per path, up to 64 Mi paths) "
          "and the atlas exceed the 126 MB L2; BVH nodes + triangles (%.0f MB) %s" %
          ((sa.bvh.shape[0] * 0.5 * 64 + sa.n_tris * 48) / 1e6,
           "stay L2-resident inside a step by design" if args.config != 5 else
           "exceed the L2, but its hot upper levels stay resident (ncu: 94 % L2 hit rate, 1.8 % DRAM throughput)"))
    return {
        "workload": "BASELINE %s; %d triangles, %d BVH nodes, procedural 2048x1024 RGBE env with sun, %d-layer %dx%d atlas"
                    % (cfg["name"], sa.n_tris, sa.bvh.shape[0], sa.atlas.shape[0], sa.atlas.shape[1], sa.atlas.shape[1]),
        "baseline_config": args.config,
        "resolution": [args.width, args.height], "spp_per_step": args.spp, "triangles": int(sa.n_tris),
        "bvh_nodes": int(sa.bvh.shape[0]),
        "anyhit": "shadow rays and last-bounce continuation rays stop at their first intersection (identical image; "
                  "roofline bytes count the node/leaf visits actually executed)",
        "parallelism": parallelism,
        "l2": l2,
    }


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(device), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1])); pw.append(float(r[2]))
                for n, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


def measured_hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic(config):
    """dram bytes per k_trace launch from the committed ncu --set full capture of this config, if one was recorded."""
    p = os.path.join(ROOT, "profiles", "trace_kernel_ncu.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            per = d.get("per_config", {}).get(str(config))
            if per:
                return per.get("dram_bytes_per_launch")
            if config == 2:
                return d.get("dram_bytes_per_launch")
        except Exception:
            pass
    return None


def algorithmic_bytes(st):
    # SURVEY.md section 8(d): B_ray = 60*V + 144*L + 32 in reference-layout bytes
    return 60 * st["node_visits"] + 144 * st["leaf_visits"] + 32 * st["rays"]


def find_browser():
    """BASELINE.md section 2: the preferred CPU baseline is the unmodified reference in headless Chromium on SwiftShader.
    Probed at run time; this image has none (and no network to fetch one)."""
    for name in ("chromium", "chromium-browser", "google-chrome", "google-chrome-stable", "chrome", "headless_shell"):
        p = shutil.which(name)
        if p:
            return p
    return os.environ.get("FSPT_BROWSER") or None


def run_reference(args, rank):
    """--impl reference: the reference's own algorithm on the host CPU, all host threads, one 1-spp pass per step.
    In order of preference: (1) the unmodified reference in headless Chromium on SwiftShader
    (oracle/swiftshader/run_harness.py), when a browser AND a copy of the reference are present at run time -- neither
    exists on the GPU box (probed below); (2) the reference's own camera.fs + tracer.fs compiled for the CPU
    (oracle/_ref/libfspt_ref.so, kind "reference": built where the reference tree exists, travels with the snapshot);
    (3) the repo's C++ restatement of the shaders (kind "port").  The scene is compiled by the oracle's own host code:
    the product library is not loaded in this arm."""
    if rank != 0:
        return
    import oracle
    from fspt_b200 import scenes
    W, H = args.width, args.height
    cores = os.cpu_count() or 1
    browser, ref_root = find_browser(), os.environ.get("FSPT_REFERENCE_ROOT", "/root/reference")
    if browser and os.path.isdir(ref_root) and CONFIGS[args.config]["scene"] == "bunny":
        try:
            sys.path.insert(0, os.path.join(ROOT, "oracle", "swiftshader"))
            import run_harness
            r = run_harness.time_reference(browser, ref_root, W, H, args.steps, args.warmup)
            val = args.steps * W * H / r["seconds"] / 1e6
            print(json.dumps({
                "impl": "reference", "metric": METRIC, "value": val, "unit": "Mpath-samples/s", "n_gpus": args.gpus,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["seconds"] / args.steps * 1e3,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": {"workload": "unmodified reference shaders, headless Chromium + SwiftShader, scene/bunny.json "
                                       "with the missing blobs substituted, %dx%d" % (W, H)},
                "cpu_baseline": {"value": val, "unit": "Mpath-samples/s", "cores": cores, "kind": "reference",
                                 "sample": "%d x (drawCamera + drawTracer) passes, gl.finish-bracketed" % args.steps},
                "e2e": {"value": val, "unit": "Mpath-samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            }))
            return
        except Exception as e:  # fall through to the port, say why
            sys.stderr.write("SwiftShader harness failed (%s); timing the CPU build of the shaders instead\n" % e)
    oracle.build()
    sa, cam = build_scene(args, host=oracle if CONFIGS[args.config]["scene"] == "bunny" else None)
    tracer, camera, kind = cpu_path(sa)
    rc, rt = scenes.rand_bases(args.steps + args.warmup + 1, 1)
    lens = scenes.lens_features(cam)

    def one(k, trace=None, cam_fn=None):
        pos, d = (cam_fn or camera)(W, H, cam["eye"], cam["dir"], cam["fov_scale"], lens, rc[k])
        (trace or tracer)(pos, d, W, H, k, rt[k], cam["env_theta"])
    for k in range(args.warmup):
        one(k)
    t0 = time.perf_counter()
    for k in range(args.steps):
        one(args.warmup + k)
    dt = time.perf_counter() - t0
    val = args.steps * W * H / dt / 1e6
    sample = "%d x (drawCamera + drawTracer) 1-spp passes of the %dx%d frame (of %d spp)" % (args.steps, W, H, args.spp)
    base = {"value": val, "unit": "Mpath-samples/s", "cores": cores, "kind": kind, "sample": sample,
            "what": CPU_KINDS[kind],
            "browser_probe": browser or "none found (chromium / google-chrome / chrome / headless_shell)"}
    if kind == "reference":  # the repo's restatement beside it, one pass: it is the faster of the two
        O = oracle.Oracle(sa)
        t1 = time.perf_counter()
        one(args.warmup + args.steps, trace=O.trace, cam_fn=oracle.camera)
        base["port_value"] = W * H / (time.perf_counter() - t1) / 1e6
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": val, "unit": "Mpath-samples/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, sa, 1, "host CPU, %d threads" % cores),
        "cpu_baseline": base,
        "e2e": {"value": val, "unit": "Mpath-samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


CPU_KINDS = {
    "reference": "the reference's own camera.fs + tracer.fs, compiled for the CPU from /root/reference/shader by "
                 "`make -C oracle ref` (oracle/_ref/libfspt_ref.so, prebuilt where the reference tree exists), all host threads",
    "port": "oracle/fspt_oracle.cpp, the repo's C++ restatement of the shaders (oracle/_ref was not shipped with this "
            "snapshot), all host threads",
}


def cpu_path(sa):
    """(trace, camera, kind) of the CPU baseline: the reference's shaders compiled for the CPU when that library is
    present (it is built where /root/reference exists and travels with the snapshot), else the oracle port."""
    import oracle
    from oracle import reference_shaders
    if reference_shaders.available():
        return reference_shaders.Reference(sa).trace, reference_shaders.camera, "reference"
    return oracle.Oracle(sa).trace, oracle.camera, "port"


def verify_parity(rank, world, local_rank, comm_ok):
    """A 96x64 frame, 8 samples, through the same path as the benchmark (rank 0 uploads, fspt_scene_broadcast,
    tiles x sample sets, fspt_reduce_accum) against the CPU oracle, bit for bit.  Returns (ok, what) on rank 0."""
    from fspt_b200 import capi, scenes, dist as fdist
    W, H, N = 96, 64, 8
    sa, cam = scenes.bunny_class(subdiv=3, atlas_res=32, env_size=(128, 64))
    ctx = capi.Context(W, H, local_rank)
    try:
        if world > 1:
            fdist.init_comm(ctx, rank, world)
            if rank == 0:
                ctx.scene_upload(sa)
            ctx.scene_broadcast(0)
        else:
            ctx.scene_upload(sa)
        ctx.set_accum_mode(1)
        rc, rt = scenes.rand_bases(N, 21)
        fr = ctx.frame(cam["eye"], cam["dir"], cam["fov_scale"], scenes.lens_features(cam), cam["env_theta"])
        n_tiles = max(1, world // 2) if world % 2 == 0 else 1  # two sample sets per tile: a two-term f32 sum is order-free
        rect, ticks = fdist.partition(rank, world, W, H, N, n_tiles=n_tiles)
        ctx.set_tile(*rect)
        ctx.clear()
        ctx.render(fr, 0, rc[ticks], rt[ticks])
        if world > 1:
            ctx.reduce_accum(0)
        got = ctx.read_accum()
    finally:
        ctx.close()
    if rank != 0:
        return None, None
    import oracle
    oracle.build()
    O = oracle.Oracle(sa)
    cols = []
    for k in range(N):
        pos, d = oracle.camera(W, H, cam["eye"], cam["dir"], cam["fov_scale"], scenes.lens_features(cam), rc[k])
        _, col, _ = O.trace(pos, d, W, H, 0, rt[k], cam["env_theta"], want_color=True)
        cols.append(col[..., :3])
    # the association the partition implies: per tile, sum over its sample sets of (sequential sum of that set's ticks)
    n_sets = world // n_tiles
    ref = np.zeros((H, W, 3), np.float32)
    for t in range(n_tiles):
        (x0, y0, w, h), _ = fdist.partition(t * n_sets, world, W, H, N, n_tiles=n_tiles)
        tile = None
        for s in range(n_sets):
            part = np.zeros((h, w, 3), np.float32)
            for k in fdist.shard_ticks(N, s, n_sets):
                part = part + cols[k][y0:y0 + h, x0:x0 + w]
            tile = part if tile is None else tile + part
        ref[y0:y0 + h, x0:x0 + w] = tile
    ok = bool(np.array_equal(got[..., :3].view(np.uint32), ref.view(np.uint32)) and np.all(got[..., 3] == N))
    return ok, "96x64, 8 samples, %d tile(s) x %d sample set(s), accumulation sum bit-exact vs CPU oracle" % (n_tiles, n_sets)


DUMP_LIMIT = 64 * 10 ** 6  # bytes written by --dump-outputs, .npy headers included


def dump_outputs(out_dir, accum):
    """--dump-outputs: the (H, W, 4) float32 accumulation buffer the timed render left, as a caller of fspt_read_accum
    receives it, so that two builds can be compared output for output.  A buffer above 64 MB (config 5) is replaced by
    a fixed, seeded sample of its pixels, accum.npy (n, 4), with their row-major pixel indices in accum_pixel_index.npy."""
    os.makedirs(out_dir, exist_ok=True)
    px = accum.reshape(-1, 4)
    if accum.nbytes > DUMP_LIMIT:
        n = (DUMP_LIMIT - 1024) // (px.itemsize * 4 + 8)
        idx = np.sort(np.random.default_rng(0).choice(px.shape[0], n, replace=False))
        np.save(os.path.join(out_dir, "accum_pixel_index.npy"), idx.astype(np.float64))
        accum = px[idx]
    np.save(os.path.join(out_dir, "accum.npy"), np.ascontiguousarray(accum, np.float32))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=sorted(CONFIGS))
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--tiles", type=int, default=None, help="strong scaling: number of image tiles (default: automatic)")
    ap.add_argument("--width", type=int, default=None)
    ap.add_argument("--height", type=int, default=None)
    ap.add_argument("--spp", type=int, default=None)
    ap.add_argument("--subdiv", type=int, default=6)
    ap.add_argument("--atlas-res", type=int, default=2048)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-verify", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the accumulation buffer of the last one to DIR/accum.npy (float32)")
    args = ap.parse_args()
    cfg = CONFIGS[args.config]
    args.width = args.width or cfg["res"][0]
    args.height = args.height or cfg["res"][1]
    args.spp = args.spp or cfg["spp"]

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    if args.warmup < 3:
        args.warmup = 3

    import torch
    import torch.distributed as dist
    from fspt_b200 import scenes
    from fspt_b200.path_tracer import PathTracer
    from fspt_b200 import dist as fdist

    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        fdist.share_host_threads()  # (measured at N = 2 on a 24-core host: rank 0 staging with all 24 threads instead of its
                                    # 12 made the e2e step 30.9 ms instead of 29.7 -- the other rank's process needs cores too)

    parity = None
    if not args.no_verify:
        parity = verify_parity(rank, world, local_rank, True)

    # the scene is compiled (BVH build, atlas packing) by ONE process per box; the other ranks receive the device-resident
    # records over NVLink (fspt_scene_broadcast), exactly like the e2e path below
    W, H, spp = args.width, args.height, args.spp
    sa, cam = build_scene(args) if rank == 0 else (None, None)
    if world > 1:
        box = [cam]
        dist.broadcast_object_list(box, src=0)  # the camera dict only
        cam = box[0]
    pt = PathTracer(sa, (W, H), cam, device=local_rank)
    ctx = pt.ctx
    if world > 1:
        fdist.init_comm(ctx, rank, world)   # NCCL communicator inside the library (C ABI)
        ctx.scene_broadcast(0)
        ctx.set_accum_mode(1)               # f32 sum + per-pixel sample count, reduced over NVLink
    if args.scaling == "strong":
        # ONE frame of `spp` samples split over the ranks: tiles x sample sets
        rect, ticks = fdist.partition(rank, world, W, H, spp, n_tiles=args.tiles)
        n_tiles, n_sets = fdist.tile_grid(world, W, H, args.tiles)
        rc_all, rt_all = scenes.rand_bases(spp, 1)
        parallelism = "strong scaling: %d tile(s) x %d sample set(s), ncclReduce(sum) behind the C ABI" % (n_tiles, n_sets)
        samples_per_step = float(W) * H * spp
    else:
        # rank r renders ticks r, r+G, ... of a (G*spp)-sample frame: its own rand-base entries (SURVEY 8e)
        rect, ticks = (0, 0, W, H), fdist.shard_ticks(world * spp, rank, world)
        rc_all, rt_all = scenes.rand_bases(world * spp, 1)
        parallelism = "weak scaling: sample-set sharding x%d (%d spp per GPU), ncclReduce(sum) behind the C ABI" % (world, spp)
        samples_per_step = float(W) * H * spp * world
    ctx.set_tile(*rect)
    rc, rt = rc_all[ticks].copy(), rt_all[ticks].copy()
    flush = torch.empty(512 << 20, dtype=torch.uint8, device="cuda")
    out8 = np.empty((H, W, 4), np.uint8)

    def barrier():
        ctx.synchronize()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def step():
        """clear + this rank's samples (+ reduce), all enqueued on the library's stream.  Returns (device ms, stats)."""
        pt.clear()
        if len(rc):
            ctx.render(pt._frame(), 0, rc, rt)
        if world > 1:
            ctx.reduce_accum(0)
        st = pt.stats()  # synchronises the library stream; render_ms / trace_ms / reduce_ms are CUDA-event times on it
        ms = (st["render_ms"] if len(rc) else 0.0) + (st["reduce_ms"] if world > 1 else 0.0)
        return ms, st

    for w in range(args.warmup):
        if w == 0 and world > 1 and not args.no_e2e:
            # the e2e path's collectives are warmed up too: NCCL sets a communicator's channels up lazily, at the first
            # call of each collective (measured: 290-380 ms for the first ncclBroadcast, 0.5 ms afterwards)
            if rank == 0:
                ctx.scene_upload(sa)
            ctx.scene_broadcast(0)
        step()
        if rank == 0:
            pt.drawQuad(out8)
    barrier()
    sampler = ClockSampler(local_rank) if rank == 0 else None
    launches0 = pt.stats()["kernel_launches"]
    dev_ms, trace_ms, shade_ms, alg_bytes, rays, primary_ms = 0.0, 0.0, 0.0, 0, 0, 0.0
    t_wall0 = time.perf_counter()
    for _ in range(args.steps):
        flush.fill_(1)  # L2 flush between timed iterations (outside the event-timed region)
        torch.cuda.synchronize()
        ms, st = step()
        dev_ms += ms
        trace_ms += st["trace_ms"]
        shade_ms += st["shade_ms"]
        primary_ms += st.get("primary_trace_ms", 0.0)
        rays += st["last_rays"]
        alg_bytes += algorithmic_bytes({"node_visits": st["last_node_visits"], "leaf_visits": st["last_leaf_visits"],
                                        "rays": st["last_rays"]})
    barrier()
    wall_ms = (time.perf_counter() - t_wall0) * 1e3
    launches = pt.stats()["kernel_launches"] - launches0
    clocks = sampler.stop() if sampler else None
    t = torch.tensor([dev_ms, float(rays)], dtype=torch.float64, device="cuda")
    if world > 1:
        tmax = t.clone()
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        tsum = t.clone()
        dist.all_reduce(tsum, op=dist.ReduceOp.SUM)
        dev_ms_max, rays_total = float(tmax[0]), float(tsum[1])
    else:
        dev_ms_max, rays_total = dev_ms, float(rays)
    value = samples_per_step * args.steps / (dev_ms_max * 1e-3) / 1e6
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, ctx.read_accum())  # before the e2e steps below render into the same buffer

    # ---- end-to-end through the host API with host buffers ---------------------------------------------------
    e2e = None
    if not args.no_e2e:
        n_e2e = max(1, min(args.steps, 5))
        h2d = 0

        def e2e_step():
            nonlocal h2d
            if rank == 0:
                # host buffers -> HBM, once per box.  fspt_scene_upload_async: the call returns when everything but the
                # atlas has been consumed; the atlas is staged + DMA'd by the context's thread while the primary traversal
                # of the render below already runs (the library waits for it before its first shading launch)
                h2d = ctx.scene_upload(sa, wait=False) + 2 * 4 * len(rc)
            if world > 1:
                ctx.scene_broadcast(0)                         # device -> device over NVLink
            step()
            if rank == 0:
                pt.drawQuad(out8)  # post-pass + D2H of the RGBA8 frame
        # The step's inputs lie in pinned host memory: the two large byte buffers of the scene (atlas, environment) are
        # page-locked once, in place (fspt_host_register) -- the library then DMAs them from where they lie; the geometry
        # buffers are repacked through the library's own pinned staging whatever memory they come from.
        pinned = []
        if rank == 0:
            from fspt_b200 import capi
            for a in (sa.atlas, sa.env):
                if a.flags["C_CONTIGUOUS"] and a.dtype == np.uint8:
                    pinned.append(capi.host_register(a))
        e2e_step()  # one untimed pass: the staging threads and pinned blocks of the upload path are warm
        barrier()
        t0 = time.perf_counter()
        for _ in range(n_e2e):
            e2e_step()
        barrier()
        e2e_s = time.perf_counter() - t0
        if rank == 0:
            ctx.upload_wait()
            for a in pinned:
                capi.host_unregister(a)
        e2e = {"value": n_e2e * samples_per_step / e2e_s / 1e6, "unit": "Mpath-samples/s",
               "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(W * H * 4), "steps": n_e2e,
               "h2d_note": "size of the host buffers handed to fspt_scene_upload_async; constant-colour atlas layers are "
                           "recognised on the host and do not cross PCIe",
               "ms_per_step": e2e_s / n_e2e * 1e3,
               "includes": "fspt_scene_upload_async on rank 0 (all scene buffers from host, atlas + environment page-locked in place; the atlas transfer overlaps the primary traversal)%s + clear + render + "
                           "ncclReduce + post-pass + RGBA8 read-back" % (" + fspt_scene_broadcast to the other ranks" if world > 1 else "")}

    if rank == 0:
        hbm_peak, hbm_src = measured_hbm_peak()
        achieved = alg_bytes / (trace_ms * 1e-3) / 1e9 if trace_ms > 0 else 0.0
        # the ceiling that applies to an L2-resident BVH: streaming reads over a 32 MB buffer, measured live
        try:
            l2_gbs = max(ctx.debug_read_bandwidth(32 << 20, 200) for _ in range(3))
            hbm_read_gbs = ctx.debug_read_bandwidth(4 << 30, 4)
        except Exception:
            l2_gbs = hbm_read_gbs = None
        # Every configuration is served by L1/L2, not HBM: the BVH of configs 1-4 fits the 126 MB L2, and for config 5
        # (0.7 GB of nodes + triangles) ncu measures a 94 % L2 hit rate and 1.8 % DRAM throughput in the bounce launches
        # (profiles/r02_k_trace_c5_ncu.txt) -- the hot upper levels stay resident.  Algorithmic bytes over the HBM copy
        # peak would read 1.26-1.44, i.e. HBM is not the bound; the ceiling that applies is L2->SM.
        if l2_gbs:
            bound, peak, peak_src = "l2", l2_gbs, ("measured live: fspt_debug_read_bandwidth over 32 MB (L1-bypassing 16-byte "
                                                   "loads, persistent grid) = the L2->SM read ceiling SURVEY 8d names for an "
                                                   "L2-served BVH")
        else:
            bound, peak, peak_src = "hbm", hbm_peak, hbm_src
        line = {
            "metric": METRIC, "value": value, "unit": "Mpath-samples/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dev_ms_max / args.steps, "higher_is_better": True,
            "scaling": args.scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "mrays_per_s": rays_total / (dev_ms_max * 1e-3) / 1e6,
            "wall_ms_per_step": wall_ms / args.steps,
            "config": workload_config(args, sa, world, parallelism),
            "clocks": clocks, "gpu_launches": int(launches),
            "roofline": {
                "bound": bound, "kernel": "k_trace (BVH traversal + ray-triangle)", "achieved": achieved, "peak": peak,
                "unit": "GB/s", "frac": achieved / peak if peak else None, "traffic": ncu_traffic(args.config),
                "peak_source": peak_src,
                "algorithmic_bytes": "sum over rays of 60*V + 144*L + 32 (reference-layout bytes, SURVEY 8d), V/L counted on device",
                "kernel_ms_per_step": trace_ms / args.steps, "share_of_step": trace_ms / dev_ms if dev_ms else None,
                "shade_ms_per_step": shade_ms / args.steps,
                "hbm_copy_peak": hbm_peak, "frac_of_hbm_copy_peak": achieved / hbm_peak,
                "l2_read_peak": l2_gbs, "hbm_read_measured_here": hbm_read_gbs,
            },
        }
        if world == 1:
            # SURVEY 8d, config 3: "report primary-only (bvh_test mode) and full-path numbers" -- mode=test (main.js:882-884,
            # bvh_test.fs:224-232): one camera pass + one primary intersectScene with the visit counter per pixel, the
            # traversal launch timed with CUDA events on the library's stream (1 ray per pixel: a short launch)
            try:
                ctx.set_tile(0, 0, W, H)
                for k in range(2):
                    ctx.debug_primary(pt._frame(), float(rc_all[0]), want_rays=False)
                st0 = pt.stats()
                ctx.debug_primary(pt._frame(), float(rc_all[0]), want_rays=False)
                stp = pt.stats()
                line["primary_only"] = {
                    # inside the timed steps: the camera-fused primary launches (spp rays per pixel), CUDA-event timed
                    "in_render_mrays_per_s": (W * H * float(len(rc)) * args.steps) / (primary_ms * 1e-3) / 1e6 if primary_ms > 0 else None,
                    "in_render_ms_per_step": primary_ms / args.steps,
                    # mode=test: one ray per pixel with the exact visit counter (a short launch)
                    "mrays_per_s": W * H / (stp["trace_ms"] * 1e-3) / 1e6 if stp["trace_ms"] > 0 else None,
                    "rays": W * H, "kernel_ms": stp["trace_ms"],
                    "node_visits_per_ray": (stp["node_visits"] - st0["node_visits"]) / float(W * H),
                    "leaf_visits_per_ray": (stp["leaf_visits"] - st0["leaf_visits"]) / float(W * H),
                    "what": "fspt_debug_primary = mode=test of the reference (bvh_test.fs): camera pass + primary closest-hit "
                            "traversal with the exact visit counter, one ray per pixel"}
            except Exception as e:  # a measurement aid must not cost the bench line
                line["primary_only"] = {"error": str(e)}
        if parity is not None and parity[0] is not None:
            line["parity"] = parity[0]
            line["parity_check"] = parity[1]
        if e2e:
            line["e2e"] = e2e
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline(args, sa, cam)
        print(json.dumps(line))
    pt.close()
    if world > 1:
        dist.destroy_process_group()


def cpu_baseline(args, sa, cam):
    """The CPU implementation of the same frame on the GPU box's host cores, bounded sample: the reference's shaders
    compiled for the CPU (kind "reference") when oracle/_ref travelled with the snapshot, else the oracle (kind "port")."""
    import oracle
    from fspt_b200 import scenes
    oracle.build()
    tracer, camera, kind = cpu_path(sa)
    W, H = args.width, args.height
    cores = os.cpu_count() or 1
    rc, rt = scenes.rand_bases(64, 1)
    lens = scenes.lens_features(cam)
    n, t_total, k = 0, 0.0, 0
    while t_total < 10.0 and k < 64:
        t0 = time.perf_counter()
        pos, d = camera(W, H, cam["eye"], cam["dir"], cam["fov_scale"], lens, rc[k])
        tracer(pos, d, W, H, k, rt[k], cam["env_theta"])
        t_total += time.perf_counter() - t0
        n += 1
        k += 1
    out = {"value": n * W * H / t_total / 1e6, "unit": "Mpath-samples/s", "cores": cores, "kind": kind, "what": CPU_KINDS[kind],
           "sample": "%d of %d spp of the same %dx%d frame (%.1f s of CPU work, all %d host threads)" % (n, args.spp, W, H, t_total, cores)}
    if kind == "reference":
        O = oracle.Oracle(sa)
        t0 = time.perf_counter()
        pos, d = oracle.camera(W, H, cam["eye"], cam["dir"], cam["fov_scale"], lens, rc[0])
        O.trace(pos, d, W, H, 0, rt[0], cam["env_theta"])
        out["port_value"] = W * H / (time.perf_counter() - t0) / 1e6
    return out


if __name__ == "__main__":
    main()
