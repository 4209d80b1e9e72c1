"""Multi-GPU parity (needs >= 2 B200s on one box: `gpurun --gpus 2 -- python -m pytest tests/test_gpu_multi.py -m gpu`;
skipped on a single-GPU box; `bench.py --gpus N` repeats the same check as its "parity" key so that the driver's scaling
run records it).  Everything collective goes through the C ABI (fspt_comm_init / fspt_scene_broadcast /
fspt_reduce_accum): sample-set sharding + ncclReduce(sum) over NVLink must equal the sum of the oracle's per-sample
colours, its mean must match the reference running mean within f32 summation-order error, a scene received by
ncclBroadcast must render the same bits as one uploaded from the host, and tile sharding must assemble the frame."""
import os
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
W, H, N = 96, 64, 8


def _worker(rank, world, port, out_dir):
    sys.path.insert(0, ROOT)
    import torch
    import torch.distributed as dist
    from fspt_b200 import capi, dist as fdist, scenes
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    sa, cam = scenes.bunny_class(subdiv=3, atlas_res=32, env_size=(128, 64))
    ctx = capi.Context(W, H, rank)
    fdist.init_comm(ctx, rank, world)       # NCCL communicator inside the library
    if rank == 0:
        ctx.scene_upload(sa)                # only rank 0 touches the host buffers ...
    ctx.scene_broadcast(0)                  # ... the other rank receives the device-resident records over NVLink
    ctx.set_accum_mode(1)
    rc, rt = scenes.rand_bases(N, 21)
    fr = ctx.frame(cam["eye"], cam["dir"], cam["fov_scale"], scenes.lens_features(cam), cam["env_theta"])
    # (1) sample-set sharding
    ticks = fdist.shard_ticks(N, rank, world)
    ctx.clear()
    ctx.render(fr, 0, rc[ticks], rt[ticks])
    ctx.reduce_accum(0)                     # enqueued on the library's stream; read_accum synchronises
    if rank == 0:
        np.save(os.path.join(out_dir, "sum.npy"), ctx.read_accum())
        np.save(os.path.join(out_dir, "rgba.npy"), ctx.resolve())
    # (2) tile sharding: rank r renders every tick of its own band
    rect, tks = fdist.partition(rank, world, W, H, N, n_tiles=world)
    ctx.set_tile(*rect)
    ctx.clear()
    ctx.render(fr, 0, rc[tks], rt[tks])
    ctx.reduce_accum(0)
    if rank == 0:
        np.save(os.path.join(out_dir, "tiles.npy"), ctx.read_accum())
    # (3) unequal sample sets (5 ticks over 2 ranks): per-pixel counts in the alpha channel keep the mean exact
    ctx.set_tile(0, 0, W, H)
    ticks5 = fdist.shard_ticks(5, rank, world)
    ctx.clear()
    ctx.render(fr, 0, rc[ticks5], rt[ticks5])
    ctx.reduce_accum(0)
    if rank == 0:
        np.save(os.path.join(out_dir, "sum5.npy"), ctx.read_accum())
    # (4) asynchronous upload on rank 0 + broadcast: the atlas part of the broadcast is deferred behind the primary
    # traversal launch of the next render on every rank; same bits as (1)
    if rank == 0:
        ctx.scene_upload(sa, wait=False)
    ctx.scene_broadcast(0)
    ctx.clear()
    ctx.render(fr, 0, rc[ticks], rt[ticks])
    ctx.reduce_accum(0)
    if rank == 0:
        np.save(os.path.join(out_dir, "sum_async.npy"), ctx.read_accum())
    # (5) a rank that renders nothing after a broadcast (1 tick over 2 ranks): its reduce issues the deferred atlas part
    if rank == 0:
        ctx.scene_upload(sa, wait=False)
    ctx.scene_broadcast(0)
    ctx.clear()
    ticks1 = fdist.shard_ticks(1, rank, world)
    if len(ticks1):
        ctx.render(fr, 0, rc[ticks1], rt[ticks1])
    ctx.reduce_accum(0)
    if rank == 0:
        np.save(os.path.join(out_dir, "sum1.npy"), ctx.read_accum())
    # (6) ... and both ranks render from that scene afterwards
    ctx.clear()
    ctx.render(fr, 0, rc[ticks], rt[ticks])
    ctx.reduce_accum(0)
    if rank == 0:
        np.save(os.path.join(out_dir, "sum_after.npy"), ctx.read_accum())
    # (7) a scene of another atlas resolution and environment size: the receiver re-creates every array (a non-power-of-
    # two environment, refractive materials); (8) the same scene with plain atlas layers on the wire: the receiver
    # switches from the interleaved array to the plain one; (9) and back.  Every rank renders all ticks of the whole frame.
    sp, cam_p = scenes.pbr_scene(atlas_res=64, subdiv=2, env_size=(96, 48))
    fr_p = ctx.frame(cam_p["eye"], cam_p["dir"], cam_p["fov_scale"], scenes.lens_features(cam_p), cam_p["env_theta"])
    ctx.set_accum_mode(0)
    for step, plain in ((7, False), (8, True), (9, False)):
        if rank == 0:
            if plain:
                os.environ["FSPT_PLAIN_ATLAS"] = "1"
            ctx.scene_upload(sp)
            os.environ.pop("FSPT_PLAIN_ATLAS", None)
        ctx.scene_broadcast(0)
        ctx.clear()
        ctx.render(fr_p, 0, rc, rt)
        np.save(os.path.join(out_dir, "step%d_rank%d.npy" % (step, rank)), ctx.read_accum())
    ctx.close()
    dist.destroy_process_group()


def test_two_gpu_sample_sharding_matches_oracle(tmp_path, oracle_mod):
    import torch
    import torch.multiprocessing as mp
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    from fspt_b200 import scenes
    mp.spawn(_worker, args=(2, 29650 + os.getpid() % 300, str(tmp_path)), nprocs=2, join=True)
    sa, cam = scenes.bunny_class(subdiv=3, atlas_res=32, env_size=(128, 64))
    O = oracle_mod.Oracle(sa)
    rc, rt = scenes.rand_bases(N, 21)
    cols, mean = [], None
    for k in range(N):
        pos, d = oracle_mod.camera(W, H, cam["eye"], cam["dir"], cam["fov_scale"], scenes.lens_features(cam), rc[k])
        _, col, _ = O.trace(pos, d, W, H, 0, rt[k], cam["env_theta"], want_color=True)
        cols.append(col[..., :3])
        mean = cols[k] if mean is None else (cols[k] + mean * np.float32(k)) / np.float32(k + 1)
    z = np.zeros_like(cols[0])
    ref = ((((z + cols[0]) + cols[2]) + cols[4]) + cols[6]) + ((((z + cols[1]) + cols[3]) + cols[5]) + cols[7])
    got = np.load(tmp_path / "sum.npy")[..., :3]
    assert np.array_equal(got.view(np.uint32), ref.view(np.uint32))
    assert np.allclose(got / N, mean, rtol=3e-6, atol=1e-7)
    assert np.all(np.load(tmp_path / "sum.npy")[..., 3] == N)   # per-pixel sample counts
    rgba = np.load(tmp_path / "rgba.npy")
    full = np.zeros((H, W, 4), np.float32)
    full[..., :3] = got / np.float32(N)
    assert np.abs(rgba.astype(int) - oracle_mod.draw(full).astype(int)).max() <= 1
    # tile sharding: every pixel received all N samples in tick order from ONE rank -> plain sequential sum
    seq = z.copy()
    for k in range(N):
        seq = seq + cols[k]
    tiles = np.load(tmp_path / "tiles.npy")
    assert np.array_equal(tiles[..., :3].view(np.uint32), seq.view(np.uint32)) and np.all(tiles[..., 3] == N)
    # unequal shards: ticks {0,2,4} + {1,3}
    ref5 = (((z + cols[0]) + cols[2]) + cols[4]) + ((z + cols[1]) + cols[3])
    sum5 = np.load(tmp_path / "sum5.npy")
    assert np.array_equal(sum5[..., :3].view(np.uint32), ref5.view(np.uint32)) and np.all(sum5[..., 3] == 5)
    # asynchronous upload + two-phase broadcast: same bits; a rank that only reduces; rendering afterwards
    first = np.load(tmp_path / "sum.npy")
    assert np.array_equal(np.load(tmp_path / "sum_async.npy").view(np.uint32), first.view(np.uint32))
    sum1 = np.load(tmp_path / "sum1.npy")
    assert np.array_equal(sum1[..., :3].view(np.uint32), (z + cols[0]).view(np.uint32)) and np.all(sum1[..., 3] == 1)
    assert np.array_equal(np.load(tmp_path / "sum_after.npy").view(np.uint32), first.view(np.uint32))
    # a received scene renders the bits of the uploaded one: new array shapes, plain atlas layers, interleaved again
    # (the plain and the interleaved atlas sample the same bits, test_gpu_api.py::test_plain_atlas_fallback_is_bit_identical)
    step7 = np.load(tmp_path / "step7_rank0.npy")
    assert float(step7[..., :3].max()) > 0.0
    for step in (7, 8, 9):
        r0, r1 = np.load(tmp_path / ("step%d_rank0.npy" % step)), np.load(tmp_path / ("step%d_rank1.npy" % step))
        assert np.array_equal(r0.view(np.uint32), r1.view(np.uint32)), step
        assert np.array_equal(r0.view(np.uint32), step7.view(np.uint32)), step
