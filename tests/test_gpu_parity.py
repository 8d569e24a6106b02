"""Parity tests proper: the sm_100a CUDA path, called through the C ABI, against the CPU oracle on the
same inputs.  The bar is bit-exact packed pixels (integer output; strict-f32 arithmetic on both sides);
the float framebuffer extension is checked to 1e-4 relative (BASELINE.json) and, in fact, exactly."""
import hashlib
import os
import subprocess

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KERNELS = ["mega", "persistent", "wavefront", "warpqueue", "streamqueue", "lanewalk"]


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a, dtype="<i4").tobytes()).hexdigest()


def gpu_frame(R, name, h, w, kernel="auto", spp=1, n=None, seed=1, **tuning):
    with R.Context(kernel=kernel, **tuning) as ctx:
        sc = ctx.scene(name, n=n, seed=seed)
        pr = ctx.prepare_scene(h, w, sc)
        img = ctx.render(h, w, pr, spp=spp if spp != 1 else None)
        ctx.sync()
        out = img.values()
        img.free(); pr.free(); sc.free()
    return out


def assert_same(got, want, what):
    bad = int((got != want).sum())
    if bad:
        d = np.abs(((got[..., None] >> np.array([16, 8, 0])) & 255) - ((want[..., None] >> np.array([16, 8, 0])) & 255)).max()
        raise AssertionError(f"{what}: {bad} of {got.size} pixels differ (max channel delta {d})")


@pytest.mark.parametrize("kernel", KERNELS)
@pytest.mark.parametrize("name", ["rgbbox", "irreg"])
def test_golden_png_500(R, golden, name, kernel):
    """GPU output == the reference's own rgbbox.png / irreg.png (500x500)."""
    want, _ = golden[f"{name}_500"]
    assert_same(gpu_frame(R, name, 500, 500, kernel), want, f"{name} 500^2 {kernel} vs reference PNG")


@pytest.mark.parametrize("kernel", KERNELS)
@pytest.mark.parametrize("name,h,w", [("rgbbox", 200, 200), ("irreg", 200, 200), ("rgbbox", 37, 91), ("irreg", 130, 67),
                                      ("rgbbox", 1, 1), ("rgbbox", 3, 5), ("irreg", 4, 8)])
def test_vs_oracle_small(R, oracle, name, h, w, kernel):
    want, _, _ = oracle.render_scene(name, h, w)
    assert_same(gpu_frame(R, name, h, w, kernel), want, f"{name} {h}x{w} {kernel}")


@pytest.mark.parametrize("name,sha256", [("rgbbox", "723bbc1045e5ccde39a0c7e828635e3ced3ddac86abd2381da6a75a830cf9535"),
                                         ("irreg", "007736b76d3011887eb12b63b8136a827424f300f0ffb4b77f16ebf8f2b48864")])
def test_headline_1000_known_answer(R, name, sha256):
    """BASELINE.json's headline size: 1000x1000 frame hash equals the oracle/Futhark known answer."""
    for kernel in KERNELS:
        assert sha(gpu_frame(R, name, 1000, 1000, kernel)) == sha256, kernel


@pytest.mark.parametrize("kernel", KERNELS)
def test_random_scene_vs_oracle(R, oracle, kernel):
    """Config 5's generator at a size the oracle finishes quickly: deep tree, duplicate Morton codes."""
    n, h, w = 20000, 160, 200
    want, _, _ = oracle.render_scene("random", h, w, n=n, seed=1)
    assert_same(gpu_frame(R, "random", h, w, kernel, n=n, seed=1), want, f"random {n} {kernel}")


def test_random_scene_global_memory_nodes(R, oracle):
    """Tree larger than the shared-memory staging budget: exercises the mixed smem/global node fetch."""
    n, h, w = 50000, 96, 128
    want, _, _ = oracle.render_scene("random", h, w, n=n, seed=5)
    for budget in (1024, 16 * 1024, 200 * 1024):
        got = gpu_frame(R, "random", h, w, "persistent", n=n, seed=5, smem_budget=budget)
        assert_same(got, want, f"random {n} smem_budget={budget}")
    for warps, k in ((16, 2), (8, 1), (4, 2), (1, 1)):
        got = gpu_frame(R, "random", h, w, "warpqueue", n=n, seed=5, wq_warps=warps, wq_k=k)
        assert_same(got, want, f"random {n} warpqueue warps={warps} k={k}")


@pytest.mark.parametrize("kernel", KERNELS)
@pytest.mark.parametrize("name,spp", [("rgbbox", 4), ("irreg", 7)])
def test_spp_extension_vs_oracle(R, oracle, name, spp, kernel):
    h, w = 96, 128
    want, want_rgb, _ = oracle.Scene.named(name).prepare(h, w).render(h, w, spp=spp, want_rgb=True)
    with R.Context(kernel=kernel) as ctx:
        pr = ctx.prepare_scene(h, w, ctx.scene(name))
        pix, rgb = ctx.render_host(h, w, pr, spp=spp, want_rgb=True)
    assert_same(pix, want, f"{name} spp={spp} {kernel}")
    rel = np.abs(rgb - want_rgb) / np.maximum(np.abs(want_rgb), 1e-6)
    assert rel.max() <= 1e-4          # BASELINE.json's float tolerance ...
    np.testing.assert_array_equal(rgb.view(np.uint32), want_rgb.view(np.uint32))  # ... and in fact bit-exact


@pytest.mark.parametrize("tuning", [dict(wq_spread=1, wq_warps=16, wq_k=1), dict(wq_spread=1, wq_warps=3, wq_k=2),
                                    dict(wq_spread=0, wq_warps=8, wq_k=2), dict(wq_spread=1, wq_warps=24, wq_k=1), dict(wq_warps=32), dict(wq_warps=32, wq_k=2)])
def test_warpqueue_sample_spreading(R, oracle, tuning):
    """spp > 1 on the warp-queue kernel: samples of a pixel are traced by different lanes and summed in
    sample order afterwards — must be bit-identical to the sequential definition, also on partial tiles
    and in the compact (sharded) output layout."""
    import torch
    from raytracers_b200 import distributed as D
    h, w, spp = 45, 83, 5
    want, want_rgb, _ = oracle.Scene.rgbbox().prepare(h, w).render(h, w, spp=spp, want_rgb=True)
    with R.Context(kernel="warpqueue", **tuning) as ctx:
        pr = ctx.prepare_scene(h, w, ctx.rgbbox())
        pix, rgb = ctx.render_host(h, w, pr, spp=spp, want_rgb=True)
        assert_same(pix, want, f"warpqueue spread {tuning}")
        np.testing.assert_array_equal(rgb.view(np.uint32), want_rgb.view(np.uint32))
        world = 3
        padded = D.tile_layout(h, w, world)[3]
        for rank in range(world):
            tiles = torch.empty((padded, 32), dtype=torch.int32, device="cuda")
            ctx.set_shard(rank, world)
            ctx.render_shard_into(tiles.data_ptr(), h, w, pr, spp=spp)
            ctx.sync()
            np.testing.assert_array_equal(tiles.cpu().numpy(), D.extract_rank_tiles(want, rank, world))


@pytest.mark.parametrize("packet_min", [1, 8, 16, 32])
def test_warpqueue_packet_walk(R, oracle, golden, packet_min):
    """Packet steps for the dense top of the tree (wq_packet = lane threshold): same frames, bit for bit —
    reference PNG, partial tiles, spp > 1, a deep random tree (spills at arbitrary depths, drain guard), K = 2."""
    want, _ = golden["rgbbox_500"]
    assert_same(gpu_frame(R, "rgbbox", 500, 500, "warpqueue", wq_packet=packet_min), want, f"packet {packet_min} vs reference PNG")
    want, _ = golden["irreg_500"]
    assert_same(gpu_frame(R, "irreg", 500, 500, "warpqueue", wq_packet=packet_min, wq_k=2, wq_warps=12), want, f"packet {packet_min} K=2")
    w2, _, _ = oracle.Scene.rgbbox().prepare(45, 83).render(45, 83, spp=5)
    assert_same(gpu_frame(R, "rgbbox", 45, 83, "warpqueue", spp=5, wq_packet=packet_min), w2, f"packet {packet_min} spp 5")
    w3, _, _ = oracle.render_scene("random", 64, 96, n=60000, seed=3)
    assert_same(gpu_frame(R, "random", 64, 96, "warpqueue", n=60000, seed=3, wq_packet=packet_min), w3, f"packet {packet_min} deep tree")
    two = np.float32([[0, 0, 0, 1, 0, 0, 2], [3, 1, -4, 0, 1, 0, 3]])
    cam = np.float32([0, 0, 20, 0, 0, 0, 60])
    w4, _, _ = oracle.Scene.custom(two, cam).prepare(32, 48).render(32, 48)
    with R.Context(kernel="warpqueue", wq_packet=packet_min) as ctx:
        pr = ctx.prepare_scene(32, 48, ctx.scene_from_arrays(two, cam))
        assert_same(ctx.render_host(32, 48, pr), w4, f"packet {packet_min} two spheres")


@pytest.mark.parametrize("tuning", [dict(wq_warps=24), dict(wq_warps=5, wq_refill=1), dict(wq_warps=16, wq_refill=32),
                                    dict(wq_warps=8, wq_spread=0)])
def test_streamqueue_variants(R, oracle, golden, tuning):
    """K4 (continuous refill): reference PNG, partial tiles with spp > 1 (incl. the compact sharded layout), deep tree."""
    import torch
    from raytracers_b200 import distributed as D
    want, _ = golden["rgbbox_500"]
    assert_same(gpu_frame(R, "rgbbox", 500, 500, "streamqueue", **tuning), want, f"streamqueue {tuning} vs reference PNG")
    h, w, spp = 45, 83, 5
    w2, _, _ = oracle.Scene.irreg().prepare(h, w).render(h, w, spp=spp)
    with R.Context(kernel="streamqueue", **tuning) as ctx:
        pr = ctx.prepare_scene(h, w, ctx.irreg())
        assert_same(ctx.render_host(h, w, pr, spp=spp), w2, f"streamqueue {tuning} spp 5")
        world = 3
        padded = D.tile_layout(h, w, world)[3]
        for rank in range(world):
            tiles = torch.empty((padded, 32), dtype=torch.int32, device="cuda")
            ctx.set_shard(rank, world)
            ctx.render_shard_into(tiles.data_ptr(), h, w, pr, spp=spp)
            ctx.sync()
            np.testing.assert_array_equal(tiles.cpu().numpy(), D.extract_rank_tiles(w2, rank, world))
    w3, _, _ = oracle.render_scene("random", 64, 96, n=60000, seed=3)
    assert_same(gpu_frame(R, "random", 64, 96, "streamqueue", n=60000, seed=3, **tuning), w3, f"streamqueue {tuning} deep tree")


@pytest.mark.parametrize("heavy_first", [0, 1])
def test_heavy_first_claim_order_is_invisible(R, oracle, golden, heavy_first):
    """The probe pass + sorted claim order only change WHEN a tile is rendered: reference PNGs, partial tiles at
    spp > 1 (row-major and compact sharded layouts), a deep tree, pixel-bound K3 and the warp trace must all be unchanged."""
    import torch
    from raytracers_b200 import distributed as D
    for name in ("rgbbox_500", "irreg_500"):
        want, _ = golden[name]
        assert_same(gpu_frame(R, name.split("_")[0], 500, 500, "warpqueue", heavy_first=heavy_first), want, f"heavy_first={heavy_first} {name}")
    h, w, spp = 45, 83, 5
    want, want_rgb, _ = oracle.Scene.rgbbox().prepare(h, w).render(h, w, spp=spp, want_rgb=True)
    for extra in (dict(), dict(wq_spread=0), dict(wq_packet=8)):
        with R.Context(kernel="warpqueue", heavy_first=heavy_first, **extra) as ctx:
            ctx.trace_warps(True)
            pr = ctx.prepare_scene(h, w, ctx.rgbbox())
            pix, rgb = ctx.render_host(h, w, pr, spp=spp, want_rgb=True)
            assert_same(pix, want, f"heavy_first={heavy_first} {extra}")
            np.testing.assert_array_equal(rgb.view(np.uint32), want_rgb.view(np.uint32))
            t = ctx.warp_trace()
            assert t.size % 148 == 0 and (t >= 0).all() and t.max() < 1e6
            world = 3
            padded = D.tile_layout(h, w, world)[3]
            for rank in range(world):
                tiles = torch.empty((padded, 32), dtype=torch.int32, device="cuda")
                ctx.set_shard(rank, world)
                ctx.render_shard_into(tiles.data_ptr(), h, w, pr, spp=spp)
                ctx.sync()
                np.testing.assert_array_equal(tiles.cpu().numpy(), D.extract_rank_tiles(want, rank, world))
    w3, _, _ = oracle.render_scene("random", 64, 96, n=60000, seed=3)
    assert_same(gpu_frame(R, "random", 64, 96, "warpqueue", n=60000, seed=3, heavy_first=heavy_first), w3, "deep tree")
    # one tile / one pixel frames: nothing to order
    w4, _, _ = oracle.Scene.rgbbox().prepare(3, 5).render(3, 5, spp=2)
    assert_same(gpu_frame(R, "rgbbox", 3, 5, "warpqueue", spp=2, heavy_first=heavy_first), w4, "single tile")


@pytest.mark.parametrize("kernel", ["warpqueue", "lanewalk", "persistent", "mega", "wavefront", "streamqueue"])
def test_render_batch_two_frames_in_flight(R, oracle, kernel):
    """ray_b200_render_batch: frames of different scenes / sizes / spp submitted as one stream-ordered operation (two in
    flight) are bit-identical to the oracle, in the row-major and the compact shard layout, with and without float output."""
    import torch
    from raytracers_b200 import distributed as D
    cases = [("irreg", 64, 96, 5), ("rgbbox", 45, 83, 1), ("rgbbox", 45, 83, 5), ("irreg", 30, 50, 2), ("rgbbox", 8, 8, 3)]
    want = {c: getattr(oracle.Scene, c[0])().prepare(c[1], c[2]).render(c[1], c[2], spp=c[3], want_rgb=True) for c in cases}
    stream = torch.cuda.Stream()
    with torch.cuda.stream(stream), R.Context(kernel=kernel) as ctx:
        ctx.set_stream(stream.cuda_stream)
        scenes = {n: ctx.scene(n) for n in ("rgbbox", "irreg")}
        prep = {c: ctx.prepare_scene(c[1], c[2], scenes[c[0]]) for c in cases}
        for rep in range(3):  # the lanes' scratch (cursor, sample buffers) is reused across batches
            pix = {c: torch.full((c[1], c[2]), -1, dtype=torch.int32, device="cuda") for c in cases}
            rgb = {c: torch.zeros((c[1], c[2], 3), dtype=torch.float32, device="cuda") for c in cases[:3]}
            ctx.render_batch([dict(prepared=prep[c], h=c[1], w=c[2], spp=c[3], out_dev=pix[c].data_ptr(),
                                   out_rgb_dev=rgb[c].data_ptr() if c in rgb else None) for c in cases])
            got = {c: pix[c].cpu().numpy() for c in cases}  # same stream: ordered after the whole batch
            assert ctx.last_render_ms() > 0
            for c in cases:
                assert_same(got[c], want[c][0], f"batch {kernel} {c} rep {rep}")
            for c in rgb:
                np.testing.assert_array_equal(rgb[c].cpu().numpy().view(np.uint32), want[c][1].view(np.uint32))
        world = 3
        for rank in range(world):
            ctx.set_shard(rank, world)
            tiles = {c: torch.full((D.tile_layout(c[1], c[2], world)[3], 32), -1, dtype=torch.int32, device="cuda") for c in cases}
            ctx.render_batch([dict(prepared=prep[c], h=c[1], w=c[2], spp=c[3], shard_layout=True, out_dev=tiles[c].data_ptr()) for c in cases])
            for c in cases:
                np.testing.assert_array_equal(tiles[c].cpu().numpy(), D.extract_rank_tiles(want[c][0], rank, world))
        ctx.set_shard(0, 1)
        ctx.render_batch([])
        with pytest.raises(R.RayError):
            ctx.render_batch([dict(prepared=prep[cases[0]], h=64, w=96, spp=1, out_dev=0)])
        with pytest.raises(R.RayError):
            ctx.render_batch([dict(prepared=prep[cases[0]], h=64, w=96, spp=1, shard_layout=True, out_dev=pix[cases[0]].data_ptr(),
                                   out_rgb_dev=rgb[cases[0]].data_ptr())])


def test_render_batch_headline_frames(R):
    """1000x1000 64 spp rgbbox + irreg as one batch == the same frames rendered one by one."""
    import torch
    with R.Context() as ctx:
        prep = {n: ctx.prepare_scene(1000, 1000, ctx.scene(n)) for n in ("irreg", "rgbbox")}
        solo = {}
        for n in prep:
            solo[n] = torch.empty((1000, 1000), dtype=torch.int32, device="cuda")
            ctx.render_into(solo[n].data_ptr(), 1000, 1000, prep[n], spp=64)
        both = {n: torch.empty((1000, 1000), dtype=torch.int32, device="cuda") for n in prep}
        for _ in range(2):
            ctx.render_batch([dict(prepared=prep[n], h=1000, w=1000, spp=64, out_dev=both[n].data_ptr()) for n in prep])
        ctx.sync()
        for n in prep:
            assert torch.equal(solo[n], both[n]), n


def test_warpqueue_deep_tree_and_many_samples(R, oracle):
    """Deep tree (bigger per-warp stacks -> fewer warps fit) and a sample count larger than one ring round."""
    n, h, w = 150000, 64, 96
    want, _, _ = oracle.render_scene("random", h, w, n=n, seed=11)
    with R.Context(kernel="warpqueue") as ctx:
        pr = ctx.prepare_scene(h, w, ctx.scene_random(n, 11))
        assert pr.info()["max_depth"] >= 20
        assert_same(ctx.render_host(h, w, pr), want, "deep tree, 1 spp")
    h, w, spp = 24, 40, 300
    want, _, _ = oracle.Scene.irreg().prepare(h, w).render(h, w, spp=spp)
    with R.Context(kernel="warpqueue") as ctx:
        pr = ctx.prepare_scene(h, w, ctx.irreg())
        assert_same(ctx.render_host(h, w, pr, spp=spp), want, "300 spp, spread")



@pytest.mark.parametrize("tuning", [dict(), dict(lw_slots=32), dict(lw_slots=64, lw_warps=20), dict(lw_warps=1, lw_slots=40), dict(lw_warps=7, lw_idle_min=1),
                                    dict(lw_idle_min=32, lw_passes=1), dict(lw_passes=8, lw_slots=56, lw_warps=24), dict(wq_spread=0)])
def test_lanewalk_variants(R, oracle, golden, tuning):
    """K5 (lane-owned traversals, slot lists, dense shading batches): reference PNGs, partial tiles at spp > 1 with the float
    framebuffer, the compact sharded layout, a deep tree with duplicate Morton codes, equal-t ties, a sample count larger
    than a ring round - over slot counts, warp counts and the shading / refill thresholds.  wq_spread=0 at spp > 1 must
    fall back to the warp-queue kernel (K5 only runs spread or 1-spp frames) and still be exact."""
    import torch
    from raytracers_b200 import distributed as D
    for name in ("rgbbox_500", "irreg_500"):
        want, _ = golden[name]
        assert_same(gpu_frame(R, name.split("_")[0], 500, 500, "lanewalk", **tuning), want, f"lanewalk {tuning} {name} vs reference PNG")
    h, w, spp = 45, 83, 5
    want, want_rgb, _ = oracle.Scene.rgbbox().prepare(h, w).render(h, w, spp=spp, want_rgb=True)
    with R.Context(kernel="lanewalk", **tuning) as ctx:
        pr = ctx.prepare_scene(h, w, ctx.rgbbox())
        pix, rgb = ctx.render_host(h, w, pr, spp=spp, want_rgb=True)
        assert_same(pix, want, f"lanewalk {tuning} spp 5")
        np.testing.assert_array_equal(rgb.view(np.uint32), want_rgb.view(np.uint32))
        world = 3
        padded = D.tile_layout(h, w, world)[3]
        for rank in range(world):
            tiles = torch.empty((padded, 32), dtype=torch.int32, device="cuda")
            ctx.set_shard(rank, world)
            ctx.render_shard_into(tiles.data_ptr(), h, w, pr, spp=spp)
            ctx.sync()
            np.testing.assert_array_equal(tiles.cpu().numpy(), D.extract_rank_tiles(want, rank, world))
    w3, _, _ = oracle.render_scene("random", 64, 96, n=60000, seed=3)
    assert_same(gpu_frame(R, "random", 64, 96, "lanewalk", n=60000, seed=3, **tuning), w3, f"lanewalk {tuning} deep tree")
    w4, _, _ = oracle.Scene.irreg().prepare(24, 40).render(24, 40, spp=300)
    assert_same(gpu_frame(R, "irreg", 24, 40, "lanewalk", spp=300, **tuning), w4, f"lanewalk {tuning} 300 spp")
    w5, _, _ = oracle.Scene.rgbbox().prepare(3, 5).render(3, 5, spp=2)
    assert_same(gpu_frame(R, "rgbbox", 3, 5, "lanewalk", spp=2, **tuning), w5, "single tile")


def test_lanewalk_deep_tree_and_trace(R, oracle):
    """150 K random spheres (tree depth >= 20: deeper private stacks, fewer slots fit) and the warp-exit trace."""
    n, h, w = 150000, 64, 96
    want, _, _ = oracle.render_scene("random", h, w, n=n, seed=11)
    with R.Context(kernel="lanewalk") as ctx:
        ctx.trace_warps(True)
        pr = ctx.prepare_scene(h, w, ctx.scene_random(n, 11))
        assert pr.info()["max_depth"] >= 20
        assert_same(ctx.render_host(h, w, pr), want, "lanewalk deep tree, 1 spp")
        t = ctx.warp_trace()
        assert t.size % 148 == 0 and (t >= 0).all() and t.max() < 1e6



@pytest.mark.parametrize("kernel", ["warpqueue", "lanewalk", "mega"])
def test_peer_frame_renderer_on_one_gpu(R, oracle, kernel):
    """The fused render+gather protocol (include/ray_b200.h "peer-memory frames") with the "ranks" emulated as contexts of
    one process on one GPU: every rank writes its own pixels straight into rank 0's row-major frame slot, the last warp of
    each kernel bumps the slot's done flag, rank 0's copy stream waits for world x uses, copies out and acknowledges.  More
    frames than ring slots (back-pressure through the ack flags); frames must equal the oracle's."""
    import torch
    from raytracers_b200 import distributed as D
    h, w, world = 45, 83, 3
    frames = [("rgbbox", 1), ("irreg", 5), ("rgbbox", 5), ("irreg", 1), ("rgbbox", 2)]
    want = {f: getattr(oracle.Scene, f[0])().prepare(h, w).render(h, w, spp=f[1])[0] for f in frames}
    ctxs = [R.Context(kernel=kernel) for _ in range(world)]
    try:
        prep = [{n: c.prepare_scene(h, w, c.scene(n)) for n in ("rgbbox", "irreg")} for c in ctxs]
        rr = [D.PeerFrameRenderer(ctxs[0], 0, world, h, w, slots=2, same_process_base=0)]
        rr += [D.PeerFrameRenderer(ctxs[r], r, world, h, w, slots=2, same_process_base=rr[0].base) for r in range(1, world)]
        got = []
        for f in frames:                       # one frame at a time; rank order shuffled so rank 0 is not always first
            order = list(range(world)) if len(got) % 2 == 0 else list(range(world))[::-1]
            used = [rr[r].submit([(prep[r][f[0]], f[1])]) for r in order][0]   # all "ranks" first (see PeerFrameRenderer.render)
            outs = rr[0].consume(used)
            rr[0].copy_stream.synchronize()
            got.append(outs[0].numpy().copy())
        for r in rr:
            r.wait()
        for f, g in zip(frames, got):
            assert_same(g, want[f], f"peer frame {kernel} {f}")
        # two frames per batch (two in flight), then a third batch that wraps the ring
        for rep in range(2):
            pair = [frames[1], frames[2]]
            used = [rr[r].submit([(prep[r][p[0]], p[1]) for p in pair]) for r in range(world)][0]
            outs = rr[0].consume(used)
            rr[0].wait()
            for p, o in zip(pair, outs):
                assert_same(o.numpy(), want[p], f"peer frame batch {kernel} {p} rep {rep}")
        assert ctxs[0].flag_timeouts() == 0
        for r in rr[::-1]:
            r.close()
    finally:
        for c in ctxs:
            c.close()



def test_wavefront_ray_resort_is_invisible(R, oracle):
    """N4 experiment (RAY_WF_SORT): re-ordering the per-bounce ray queue by (direction octant, origin Morton code) only
    changes the ORDER rays are traced in - frames stay bit-identical (1 spp, spp > 1 with the in-order accumulator, deep tree)."""
    for name, h, w, spp, kw in (("rgbbox", 96, 128, 1, {}), ("irreg", 96, 128, 3, {}), ("random", 64, 96, 1, dict(n=60000, seed=3))):
        want, _, _ = oracle.render_scene(name, h, w, spp=spp, **kw)
        for bounces in (1, 4, 60):
            assert_same(gpu_frame(R, name, h, w, "wavefront", spp=spp, wf_sort=bounces, **kw), want, f"{name} wf_sort={bounces}")



@pytest.mark.parametrize("kernel", ["warpqueue", "lanewalk"])
def test_pipelined_submission_with_scene_reupload(R, oracle, kernel):
    """ray_b200_context_set_pipeline: frames of consecutive render_batch calls alternate between the two lanes WITHOUT a
    join, while the scenes they read are re-uploaded (device LBVH rebuilt, old block released) before every batch and one is
    freed mid-flight - the scene memory of a frame in flight must only be reclaimed after the frame (release_scene_block).
    World-1 peer-frame ring as the consumer; every delivered host frame must equal the oracle's."""
    from raytracers_b200 import distributed as D
    h, w = 64, 96
    cases = [("irreg", 3), ("rgbbox", 1), ("rgbbox", 4), ("irreg", 1)]
    want = {c: getattr(oracle.Scene, c[0])().prepare(h, w).render(h, w, spp=c[1])[0] for c in cases}
    with R.Context(kernel=kernel) as ctx:
        prep = {n: ctx.prepare_scene(h, w, ctx.scene(n)) for n in ("rgbbox", "irreg")}
        pf = D.PeerFrameRenderer(ctx, 0, 1, h, w, slots=4, pipeline=True)
        got = []
        for step in range(4):
            for n in prep:
                prep[n].reupload()
            pair = [cases[(2 * step) % 4], cases[(2 * step + 1) % 4]]
            outs = pf.render([(prep[c[0]], c[1]) for c in pair])
            if step == 2:                          # a scene that is still being rendered is freed and prepared again
                prep["irreg"].free()
                prep["irreg"] = ctx.prepare_scene(h, w, ctx.scene("irreg"))
            if step % 2 == 1:                      # ring of 4 slots, 2 frames per step: collect every second step
                pf.wait()
            got.append((pair, outs))
        pf.wait()
        for pair, outs in got[-2:]:                # the last two steps' host buffers are still intact (4 slots)
            for c, o in zip(pair, outs):
                assert_same(o.numpy(), want[c], f"pipelined {kernel} {c}")
        # strict mode again: a joined batch right after leaving the pipeline
        pf.close()
        out = ctx.render_host(h, w, prep["rgbbox"], spp=4)
        assert_same(out, want[("rgbbox", 4)], f"after pipeline {kernel}")



@pytest.mark.parametrize("long_path", [2, 12, 60])
def test_learned_claim_order_is_invisible(R, oracle, golden, long_path):
    """The first frame of a prepared scene on the context's stream records the longest path per tile, later frames claim
    the long-path tiles first (RAY_LEARN_ORDER / RAY_LONG_PATH): only WHEN a tile is rendered may change.  Reference PNGs
    (three frames each: recording, learned, learned), spp > 1 on partial tiles with the float framebuffer, a sharded
    row-major frame, a size change (new recording) and a scene re-upload (same spheres, order kept) must all stay bit-identical."""
    import torch
    for name in ("rgbbox_500", "irreg_500"):
        want, _ = golden[name]
        with R.Context(learn_order=1, long_path=long_path) as ctx:
            pr = ctx.prepare_scene(500, 500, ctx.scene(name.split("_")[0]))
            for rep in range(3):
                img = ctx.render(500, 500, pr)
                ctx.sync()
                assert_same(img.values(), want, f"learned order {name} long_path={long_path} frame {rep}")
                img.free()
    h, w, spp = 135, 203, 3
    want, want_rgb, _ = oracle.Scene.rgbbox().prepare(h, w).render(h, w, spp=spp, want_rgb=True)
    w2, _, _ = oracle.Scene.rgbbox().prepare(h, w).render(64, 96)
    with R.Context(learn_order=1, long_path=long_path) as ctx:
        pr = ctx.prepare_scene(h, w, ctx.rgbbox())
        for rep in range(3):
            pix, rgb = ctx.render_host(h, w, pr, spp=spp, want_rgb=True)
            assert_same(pix, want, f"learned order spp {spp} frame {rep}")
            np.testing.assert_array_equal(rgb.view(np.uint32), want_rgb.view(np.uint32))
        assert_same(ctx.render_host(64, 96, pr), w2, "other size: records again")
        assert_same(ctx.render_host(64, 96, pr), w2, "other size: learned")
        pr.reupload()
        assert_same(ctx.render_host(h, w, pr, spp=spp), want, "after re-upload (same spheres: the learned order is kept)")
        assert_same(ctx.render_host(h, w, pr, spp=spp), want, "after re-upload, second frame")
        ctx.set_shard(1, 3)                       # a shard's row-major frame: only this rank's tiles, twice
        for rep in range(2):
            out = torch.zeros((h, w), dtype=torch.int32, device="cuda")
            ctx.render_into(out.data_ptr(), h, w, pr, spp=spp)
            ctx.sync()
            got = out.cpu().numpy()
            tiles_x = (w + 7) // 8
            jj, ii = np.meshgrid(np.arange(h), np.arange(w), indexing="ij")
            mine = ((jj // 4) * tiles_x + ii // 8) % 3 == 1
            np.testing.assert_array_equal(got[mine], want[mine])
            assert (got[~mine] == 0).all()


def test_headline_config_64spp_kernels_agree(R):
    """BASELINE configs[1]/[2] (1000x1000, 64 spp): too slow for the CPU oracle inside a test, so the kernels
    (lane-bound K1, sample-spread K3, pixel-bound K3) are checked against each other bit-for-bit."""
    for name in ("rgbbox", "irreg"):
        a = gpu_frame(R, name, 1000, 1000, "persistent", spp=64)
        b = gpu_frame(R, name, 1000, 1000, "warpqueue", spp=64)
        c = gpu_frame(R, name, 1000, 1000, "warpqueue", spp=64, wq_spread=0)
        d = gpu_frame(R, name, 1000, 1000, "streamqueue", spp=64)
        e = gpu_frame(R, name, 1000, 1000, "lanewalk", spp=64)
        assert sha(a) == sha(b) == sha(c) == sha(d) == sha(e), name


def test_custom_scenes_edge_cases(R, oracle):
    cam = np.float32([0, 0, 20, 0, 0, 0, 60])
    cases = {
        "two spheres": np.float32([[0, 0, 0, 1, 0, 0, 2], [3, 1, -4, 0, 1, 0, 3]]),
        "coincident (equal t ties)": np.tile(np.float32([0, 0, 0, 0.9, 0.5, 0.1, 3]), (9, 1)),
        "nested + touching": np.float32([[0, 0, 0, 1, 1, 1, 5], [0, 0, 0, 1, 0, 0, 2], [7, 0, 0, 0, 0, 1, 2], [0, 7, 0, 0, 1, 0, 2]]),
    }
    # the second of the coincident spheres gets another colour: the tie must go to the lowest sorted index
    cases["coincident (equal t ties)"][1::2, 3:6] = (0.1, 0.9, 0.3)
    h, w = 48, 64
    for what, s in cases.items():
        want, _, _ = oracle.Scene.custom(s, cam).prepare(h, w).render(h, w)
        for kernel in KERNELS:
            with R.Context(kernel=kernel) as ctx:
                pr = ctx.prepare_scene(h, w, ctx.scene_from_arrays(s, cam))
                assert_same(ctx.render_host(h, w, pr), want, f"{what} {kernel}")


def test_prepare_aspect_differs_from_render_size(R, oracle):
    # prepare_scene fixes the camera aspect (ray.fut:243-244); render h w only sets the grid (ray.fut:246-247)
    pr_o = oracle.Scene.rgbbox().prepare(100, 300)
    want, _, _ = pr_o.render(64, 80)
    with R.Context() as ctx:
        pr = ctx.prepare_scene(100, 300, ctx.rgbbox())
        assert_same(ctx.render_host(64, 80, pr), want, "aspect from prepare_scene")


@pytest.mark.parametrize("name,kw", [("rgbbox", {}), ("irreg", {}), ("random", {"n": 30000, "seed": 4}), ("random", {"n": 2, "seed": 1}),
                                     ("random", {"n": 3, "seed": 2}), ("random", {"n": 1000, "seed": 8})])
def test_device_lbvh_build_is_bit_identical_to_host_and_oracle(R, oracle, name, kw):
    """prepare_scene runs on the device (bvh_build.cu): Morton keys, stable sort, Karras tree, fixed-count Jacobi refit
    and the packed layout must equal the host builder's (scene_host.cpp) and the oracle's arrays bit for bit."""
    s, c = R.host_scene(name, **kw)
    want = oracle.Scene.custom(s, c).prepare(120, 200).dump()
    host = R.host_lbvh(s)
    with R.Context() as ctx, R.Context(host_build=1) as ctx_h:
        pr = ctx.prepare_scene(120, 200, ctx.scene_from_arrays(s, c))
        pr_h = ctx_h.prepare_scene(120, 200, ctx_h.scene_from_arrays(s, c))
        got, got_h = pr.dump(), pr_h.dump()
        for k in ("morton", "perm", "left", "right", "parent"):
            np.testing.assert_array_equal(got[k], want[k], err_msg=f"device {k}")
            np.testing.assert_array_equal(got_h[k], want[k], err_msg=f"host {k}")
        np.testing.assert_array_equal(got["boxes"].view(np.uint32), want["boxes"].view(np.uint32))
        info, info_h = pr.info(), pr_h.info()
        for k in ("max_depth", "refit_sweeps", "stale_nodes"):
            assert info[k] == info_h[k] == host[k], k
        np.testing.assert_array_equal(info["root_box"].view(np.uint32), info_h["root_box"].view(np.uint32))
        np.testing.assert_array_equal(info["camera"].view(np.uint32), want["cam"].view(np.uint32))
        pk, pk_h = pr.packed(), pr_h.packed()
        for k in ("nodes", "nodes_soa", "geom", "colour"):
            np.testing.assert_array_equal(pk[k].view(np.uint32), pk_h[k].view(np.uint32), err_msg=f"packed {k}")
        assert pr.upload_bytes() == s.nbytes and pr_h.upload_bytes() == pr_h.device_bytes()


def test_degenerate_scenes_on_the_device_builder(R, oracle):
    cam = np.float32([0, 0, 20, 0, 0, 0, 60])
    same = np.tile(np.float32([1, 2, 3, 1, 1, 1, 0.5]), (37, 1))       # every Morton code equal: split purely by index
    flat = np.float32([[x, 0, z, 1, 1, 1, 0.4] for x in range(-3, 4) for z in range(-3, 4)])  # flat axis: 0/0 -> NaN -> 0
    for s in (same, flat):
        want = oracle.Scene.custom(s, cam).prepare(32, 32).dump()
        with R.Context() as ctx:
            got = ctx.prepare_scene(32, 32, ctx.scene_from_arrays(s, cam)).dump()
        for k in ("morton", "perm", "left", "right", "parent"):
            np.testing.assert_array_equal(got[k], want[k], err_msg=k)
        np.testing.assert_array_equal(got["boxes"].view(np.uint32), want["boxes"].view(np.uint32))


def test_work_counters_equal_reference_traversal(R, oracle):
    """The GPU traversal visits exactly the reference's set of boxes and leaves (roofline numerators)."""
    for name, size in (("rgbbox", 200), ("irreg", 200)):
        _, _, cnt = oracle.render_scene(name, size, size)
        with R.Context() as ctx:
            pr = ctx.prepare_scene(size, size, ctx.scene(name))
            got = ctx.count_work(size, size, pr)
        assert got["segments"] == cnt["segments"]
        assert got["box_tests"] == cnt["box_tests"]
        assert got["leaf_tests"] == cnt["leaf_tests"]
        assert got["node_steps"] < cnt["iterations"] / 2   # the stack walk needs far fewer steps than bvh_fold


def test_error_behaviour(R):
    with R.Context() as ctx:
        with pytest.raises(R.RayError, match="at least 2 spheres"):
            ctx.prepare_scene(8, 8, ctx.scene_from_arrays(np.float32([[0, 0, 0, 1, 1, 1, 1]]), np.float32([0, 0, 5, 0, 0, 0, 60])))
        assert ctx.get_error() is None          # the message is handed out once (main.c:64 protocol)
        pr = ctx.prepare_scene(8, 8, ctx.rgbbox())
        with pytest.raises(R.RayError):
            ctx.render(0, 8, pr)
        with pytest.raises(R.RayError):
            ctx.render(8, 8, pr, spp=0)
        img = ctx.render(8, 8, pr)              # context still usable after errors
        ctx.sync()
        assert img.shape == (8, 8)


def test_array_and_misc_api(R):
    """The rest of the generated-API surface: array constructors/accessors, report, cache clearing, config flags."""
    import ctypes as C
    L = R.load_library()
    cfg = L.futhark_context_config_new()
    L.futhark_context_config_set_debugging(cfg, 0)
    L.futhark_context_config_set_profiling(cfg, 1)
    L.futhark_context_config_set_logging(cfg, 0)
    L.futhark_context_config_set_device(cfg, b"#0")
    assert L.futhark_context_config_set_tuning_param(cfg, b"no_such_param", 1) == 1
    assert L.futhark_context_config_set_tuning_param(cfg, b"spp", 1) == 0
    names = [L.futhark_get_tuning_param_name(i) for i in range(L.futhark_get_tuning_param_count())] if hasattr(L, "futhark_get_tuning_param_count") else []
    ctxh = L.futhark_context_new(cfg)
    L.futhark_context_config_free(cfg)
    assert ctxh and not L.futhark_context_get_error(ctxh)
    data = np.arange(6 * 9, dtype=np.int32).reshape(6, 9)
    arr = L.futhark_new_i32_2d(ctxh, data.ctypes.data, 6, 9)
    assert arr
    shp = L.futhark_shape_i32_2d(ctxh, arr)
    assert (shp[0], shp[1]) == (6, 9)
    back = np.zeros_like(data)
    assert L.futhark_values_i32_2d(ctxh, arr, back.ctypes.data) == 0
    np.testing.assert_array_equal(back, data)
    raw = L.futhark_values_raw_i32_2d(ctxh, arr)
    assert raw
    alias = L.futhark_new_raw_i32_2d(ctxh, raw, 6, 9)     # wraps, does not own
    back2 = np.zeros_like(data)
    assert L.futhark_values_i32_2d(ctxh, alias, back2.ctypes.data) == 0
    np.testing.assert_array_equal(back2, data)
    assert L.futhark_free_i32_2d(ctxh, alias) == 0 and L.futhark_free_i32_2d(ctxh, arr) == 0
    assert L.futhark_context_clear_caches(ctxh) == 0 and L.futhark_context_sync(ctxh) == 0
    rep = L.futhark_context_report(ctxh)
    assert b"ray_b200" in C.string_at(rep)
    C.CDLL(None).free.argtypes = [C.c_void_p]
    C.CDLL(None).free(rep)
    L.futhark_context_free(ctxh)


def test_clear_caches_then_render_again(R, oracle):
    """futhark_context_clear_caches drops the grow-only scratch (sample buffers, ray queues, upload buffers); the next
    prepare_scene / render must simply grow it again."""
    h, w, spp = 33, 47, 4
    want, _, _ = oracle.Scene.rgbbox().prepare(h, w).render(h, w, spp=spp)
    for kernel in ("warpqueue", "wavefront"):
        with R.Context(kernel=kernel) as ctx:
            for _ in range(2):
                pr = ctx.prepare_scene(h, w, ctx.rgbbox())
                assert_same(ctx.render_host(h, w, pr, spp=spp), want, f"{kernel} around clear_caches")
                pr.free()
                assert ctx.lib.futhark_context_clear_caches(ctx.handle) == 0


def test_store_restore_and_reupload(R, oracle):
    h, w = 40, 56
    want, _, _ = oracle.render_scene("irreg", h, w)
    with R.Context() as ctx:
        sc = ctx.irreg()
        sc2 = ctx.restore_scene(sc.store())
        np.testing.assert_array_equal(sc.arrays()[0], sc2.arrays()[0])
        pr = ctx.prepare_scene(h, w, sc2)
        pr2 = ctx.restore_prepared_scene(pr.store())
        assert pr2.device_bytes() == pr.device_bytes() > 0
        pr2.reupload()
        assert_same(ctx.render_host(h, w, pr2), want, "restored prepared scene")


def test_torch_stream_and_device_buffers(R, oracle):
    import torch
    h, w = 72, 104
    want, _, _ = oracle.render_scene("rgbbox", h, w)
    with R.Context() as ctx:
        ctx.set_stream(torch.cuda.current_stream().cuda_stream)
        pr = ctx.prepare_scene(h, w, ctx.rgbbox())
        out = torch.zeros((h, w), dtype=torch.int32, device="cuda")
        ctx.render_into(out.data_ptr(), h, w, pr)
        torch.cuda.synchronize()
        assert_same(out.cpu().numpy(), want, "render_into on torch's stream")
        assert ctx.last_render_ms() > 0 and ctx.launch_count() >= 1


@pytest.mark.parametrize("world", [2, 3, 8])
def test_sharded_render_equals_single_gpu(R, oracle, world):
    """Every rank's tiles rendered on this one GPU, concatenated rank-major as an NCCL gather would,
    de-tiled by the CUDA kernel: must equal the unsharded frame (and the oracle) exactly."""
    import torch
    from raytracers_b200 import distributed as D
    h, w = 90, 122   # partial tiles on both edges
    want, _, _ = oracle.render_scene("irreg", h, w)
    padded = D.tile_layout(h, w, world)[3]
    gathered = torch.empty((world, padded, 32), dtype=torch.int32, device="cuda")
    with R.Context() as ctx:
        ctx.set_stream(torch.cuda.current_stream().cuda_stream)
        pr = ctx.prepare_scene(h, w, ctx.irreg())
        for rank in range(world):
            ctx.set_shard(rank, world)
            ctx.render_shard_into(gathered[rank].data_ptr(), h, w, pr)
            torch.cuda.synchronize()
            np.testing.assert_array_equal(gathered[rank].cpu().numpy(), D.extract_rank_tiles(want, rank, world))
        frame = torch.empty((h, w), dtype=torch.int32, device="cuda")
        ctx.detile(gathered.data_ptr(), frame.data_ptr(), h, w, world)
        torch.cuda.synchronize()
    assert_same(frame.cpu().numpy(), want, f"sharded world={world}")


def _device_count():
    try:
        import torch
        return torch.cuda.device_count()
    except Exception:
        return 0


@pytest.mark.skipif(_device_count() < 2, reason="needs at least 2 GPUs in this process")
def test_single_process_multi_gpu_context(R, oracle, tmp_path):
    """RAY_GPUS / tuning "gpus": ONE process (e.g. the unmodified main.c) drives several devices — scene replicated,
    tiles interleaved, shards pulled to device 0 with peer copies, de-tiled.  Frame must equal the oracle's."""
    g = min(_device_count(), 4)
    for name, h, w, spp in (("irreg", 90, 122, 1), ("rgbbox", 64, 96, 3)):
        want, _, _ = oracle.Scene.named(name).prepare(h, w).render(h, w, spp=spp)
        with R.Context(gpus=g) as ctx:
            pr = ctx.prepare_scene(h, w, ctx.scene(name))
            img = ctx.render(h, w, pr, spp=spp)
            ctx.sync()
            assert_same(img.values(), want, f"{name} gpus={g}")
            img2 = ctx.render(h, w, pr, spp=spp)      # buffers are reused across frames
            assert_same(img2.values(), want, f"{name} gpus={g} second frame")
            img.free(); img2.free(); pr.free()
    exe = os.path.join(ROOT, "oracle", "_ref", "main_ref")
    if os.path.exists(exe):
        ppm = str(tmp_path / "mg.ppm")
        r = subprocess.run([exe, "-s", "irreg", "-n", "120", "-m", "160", "-r", "2", "-f", ppm], capture_output=True, text=True,
                           env=dict(os.environ, RAY_GPUS=str(g)))
        assert r.returncode == 0, r.stderr + r.stdout
        tok = open(ppm).read().split()
        rgb = np.array(tok[4:], dtype=np.int32).reshape(120, 160, 3)
        want, _, _ = oracle.render_scene("irreg", 120, 160)
        assert_same((rgb[..., 0] << 16) | (rgb[..., 1] << 8) | rgb[..., 2], want, f"main.c RAY_GPUS={g}")


def test_reference_driver_binary_runs_against_the_library(tmp_path, oracle):
    """The reference's UNMODIFIED futhark/main.c, compiled against include/ray.h where the original project is
    checked out (oracle/_ref/main_ref, see __graft_entry__.build), run here: its PPM must equal the oracle frame."""
    exe = os.path.join(ROOT, "oracle", "_ref", "main_ref")
    if not os.path.exists(exe):
        exe = os.path.join(ROOT, "examples", "_built", "driver")
    if not os.path.exists(exe):
        pytest.skip("no prebuilt driver binary")
    ppm = str(tmp_path / "out.ppm")
    for name in ("rgbbox", "irreg"):
        r = subprocess.run([exe, "-s", name, "-n", "120", "-m", "160", "-r", "2", "-f", ppm], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr + r.stdout
        tok = open(ppm).read().split()
        assert tok[:4] == ["P3", "160", "120", "255"]
        rgb = np.array(tok[4:], dtype=np.int32).reshape(120, 160, 3)
        want, _, _ = oracle.render_scene(name, 120, 160)
        assert_same((rgb[..., 0] << 16) | (rgb[..., 1] << 8) | rgb[..., 2], want, f"main.c {name}")


def test_million_sphere_scene_kernels_and_builders_agree(R):
    """BASELINE configs[4]'s scene (1 M random spheres, tree depth ~25) is far too slow for the CPU oracle, so the two
    independent LBVH builders (device kernels vs host C++) and two independent traversals (lane-bound stack walk vs
    item queues with packet walk) are checked against each other: identical trees, identical frames."""
    n, h, w, spp = 1000000, 256, 320, 2
    with R.Context(kernel="warpqueue") as ctx, R.Context(kernel="mega", host_build=1) as ctx_h:
        pr = ctx.prepare_scene(h, w, ctx.scene_random(n, 1))
        pr_h = ctx_h.prepare_scene(h, w, ctx_h.scene_random(n, 1))
        a, b = pr.dump(), pr_h.dump()
        for k in ("morton", "perm", "left", "right", "parent"):
            np.testing.assert_array_equal(a[k], b[k], err_msg=k)
        np.testing.assert_array_equal(a["boxes"].view(np.uint32), b["boxes"].view(np.uint32))
        assert pr.info()["max_depth"] == pr_h.info()["max_depth"] >= 22
        assert pr.info()["stale_nodes"] == pr_h.info()["stale_nodes"]
        f1 = ctx.render_host(h, w, pr, spp=spp)
        f2 = ctx_h.render_host(h, w, pr_h, spp=spp)
        assert_same(f1, f2, "1M spheres: warpqueue/device build vs mega/host build")
        assert len(np.unique(f1)) > 1000


def test_large_frame_properties(R):
    """irreg at 4000x4000 (BASELINE config 4's frame size) — too slow for the CPU oracle inside a test, so
    size-independent properties: all kernels agree bit-for-bit; sub-sampling the 4000^2 render at stride 4
    is NOT required to equal 1000^2 (different u,v), but the top-left pixel and sky rows are: a row of pure
    sky has the same packed value at every size because v = (H-j)/H -> row 0 is v = 1 exactly."""
    a = gpu_frame(R, "irreg", 4000, 4000, "persistent")
    b = gpu_frame(R, "irreg", 4000, 4000, "mega")
    assert sha(a) == sha(b)
    small = gpu_frame(R, "irreg", 1000, 1000, "persistent")
    np.testing.assert_array_equal(a[0, ::4], small[0])  # row 0: v = 1, u = i/W identical for i = 4k


@pytest.mark.parametrize("mode", ["grid", "line", "plane", "huge", "cloud"])
def test_device_lbvh_on_adversarial_scenes(R, oracle, mode):
    """The device builder against the oracle on the adversarial set of tests/test_host_logic.py (duplicate keys, NaN
    Morton axes, clamping, n around powers of two), plus a render of each scene."""
    import zlib
    from test_host_logic import _adversarial_scene
    rng = np.random.default_rng(zlib.crc32(mode.encode()))
    cam = np.float32([0, 0, 50, 0, 0, 0, 60])
    with R.Context() as ctx:
        for n in (2, 3, 4, 5, 7, 8, 9, 31, 32, 33, 100, 257, 1000):
            s = _adversarial_scene(rng, n, mode)
            want_pr = oracle.Scene.custom(s, cam).prepare(16, 24)
            want = want_pr.dump()
            pr = ctx.prepare_scene(16, 24, ctx.scene_from_arrays(s, cam))
            got = pr.dump()
            for k in ("morton", "perm", "left", "right", "parent"):
                np.testing.assert_array_equal(got[k], want[k], err_msg=f"{mode} n={n} {k}")
            np.testing.assert_array_equal(got["boxes"].view(np.uint32), want["boxes"].view(np.uint32), err_msg=f"{mode} n={n} boxes")
            assert_same(ctx.render_host(16, 24, pr), want_pr.render(16, 24)[0], f"{mode} n={n} frame")
            pr.free()


@pytest.mark.parametrize("wq_low", [-1, 32, 40, 100, 100000])
def test_node_queue_pop_order_is_invisible(R, oracle, golden, wq_low):
    """The node queue of the warp-queue kernel is a ring whose batches take the OLDEST items while at most `wq_low` are queued
    and the newest above that (RAY_WQ_LOW; -1 = plain stack, values above the ring are clamped): the fold is a min, so the
    order in which (ray, node) items are processed may not change a pixel.  Reference PNGs with 32 and 64 rays per warp, the
    packet walk, spp > 1 (spread and pixel-bound samples) and the smallest ring with a deep tree (overflow guard)."""
    for name in ("rgbbox_500", "irreg_500"):
        want, _ = golden[name]
        for tuning in (dict(), dict(wq_k=1), dict(wq_k=1, wq_packet=8), dict(wq_k=2, wq_ncap=256)):
            with R.Context(kernel="warpqueue", wq_low=wq_low, **tuning) as ctx:
                pr = ctx.prepare_scene(500, 500, ctx.scene(name.split("_")[0]))
                assert_same(ctx.render_host(500, 500, pr), want, f"{name} wq_low={wq_low} {tuning}")
    h, w = 61, 83
    for name in ("rgbbox", "irreg"):
        sc = getattr(oracle.Scene, name)()
        for spp in (2, 5):
            want, _, _ = sc.prepare(h, w).render(h, w, spp=spp)
            for tuning in (dict(), dict(wq_spread=0), dict(wq_k=1, wq_packet=12)):
                with R.Context(kernel="warpqueue", wq_low=wq_low, **tuning) as ctx:
                    pr = ctx.prepare_scene(h, w, ctx.scene(name))
                    assert_same(ctx.render_host(h, w, pr, spp=spp), want, f"{name} spp={spp} wq_low={wq_low} {tuning}")
    n = 3000                                       # a deeper tree on the smallest (256-entry) ring: the overflow guard takes items one at a time
    want, _, _ = oracle.Scene.random(n, seed=7).prepare(40, 56).render(40, 56)
    with R.Context(kernel="warpqueue", wq_low=wq_low, wq_ncap=256) as ctx:
        pr = ctx.prepare_scene(40, 56, ctx.scene("random", n=n, seed=7))
        assert_same(ctx.render_host(40, 56, pr), want, f"random {n} wq_low={wq_low} ring 256")
