"""Ray queries (include/ray_b200.h "ray queries"): closest hit (objs_hit, ray.fut:76-86) and path colour (ray_colour,
ray.fut:126-148) of caller-supplied rays.  The CPU tests pin the oracle's loops over both (tests/ray_query_oracle.cpp) to
the reference's own render and to a brute-force closest-hit search; the GPU tests pin the CUDA kernel to those loops, the
golden PNGs and the renderer."""
import numpy as np
import pytest

import ray_query_oracle as Q

F = np.float32


def camera_rays(cam12, h, w, offsets=None):
    """Primary rays of an h x w frame, row-major, exactly as primary_ray (render_common.cuh) / get_ray (ray.fut:109-114)
    build them in f32: u = (i + ox) / w, v = (h - j + oy) / h, d = ((llc + u*horizontal) + v*vertical) - origin.
    offsets: None (1 spp) or the (ox, oy) of one sample."""
    c = np.asarray(cam12, F)
    i = np.arange(w, dtype=F)[None, :]
    hj = (F(h) - np.arange(h, dtype=F))[:, None]
    if offsets is None:
        u = np.broadcast_to(i / F(w), (h, w))
        v = np.broadcast_to(hj / F(h), (h, w))
    else:
        u = np.broadcast_to((i + F(offsets[0])) / F(w), (h, w))
        v = np.broadcast_to((hj + F(offsets[1])) / F(h), (h, w))
    rays = np.empty((h, w, 6), F)
    rays[..., 0:3] = c[0:3]
    for k in range(3):
        rays[..., 3 + k] = ((c[3 + k] + u * c[6 + k]) + v * c[9 + k]) - c[k]
    return rays.reshape(-1, 6)


def pack(colour):
    """colour_to_pixel (ray.fut:158-162): trunc(255.99 * c) per channel."""
    q = (F(255.99) * np.asarray(colour, F)).astype(np.int32)
    return (q[..., 0] << 16) | (q[..., 1] << 8) | q[..., 2]


def seeded_rays(spheres, n, seed):
    """A mix of rays: from around the scene towards sphere centres (mostly hits; unnormalised directions of any length),
    from inside spheres (the t_min = 0 re-intersection), and in random directions (many miss the root box)."""
    rng = np.random.default_rng(seed)
    pos, rad = spheres[:, 0:3], spheres[:, 6]
    lo, hi = pos.min(0) - 2 * rad.max(), pos.max(0) + 2 * rad.max()
    span = hi - lo
    rays = np.empty((n, 6), F)
    kind = rng.integers(0, 4, n)
    tgt = pos[rng.integers(0, len(pos), n)] + rng.normal(0, 0.3, (n, 3)) * rad.mean()
    org = lo + rng.random((n, 3)) * span * 3 - span        # around the scene, often outside the root box
    inside = rng.integers(0, len(pos), n)
    rays[:, 0:3] = np.where((kind == 1)[:, None], pos[inside] + rng.uniform(-0.5, 0.5, (n, 3)) * rad[inside, None], org)
    d = tgt - rays[:, 0:3]
    d = np.where((kind == 1)[:, None], rng.normal(size=(n, 3)), d)
    d = np.where((kind == 3)[:, None], rng.normal(size=(n, 3)), d)   # random directions
    d *= rng.choice([1e-2, 1.0, 37.0], n)[:, None]                    # not normalised
    rays[:, 3:6] = d
    return rays


def brute_force_objs_hit(oracle, perm, spheres, ray):
    """objs_hit without the tree: closest_hit over every leaf in Morton-sorted order (perm[leaf] = scene index; strict `<`,
    so the lowest leaf wins a tie), then the (0, t + 1) re-intersection — all through oracle_sphere_hit.
    Returns (index, t, pn, tied)."""
    import ctypes as C
    L = oracle.lib()
    out = np.empty(10, F)
    r = np.ascontiguousarray(ray, F)
    rp, op = r.ctypes.data_as(C.c_void_p), out.ctypes.data_as(C.c_void_p)
    acc_j, acc_t, ts = -1, F(1e9), []
    for k, s in enumerate(perm):
        sp = spheres[s].ctypes.data_as(C.c_void_p)
        if L.oracle_sphere_hit(sp, rp, F(0.1), acc_t, op):
            acc_j, acc_t = k, F(out[0])
        if L.oracle_sphere_hit(sp, rp, F(0.1), F(1e9), op):
            ts.append(F(out[0]))
    if acc_j < 0 or not L.oracle_sphere_hit(spheres[perm[acc_j]].ctypes.data_as(C.c_void_p), rp, F(0.0), F(acc_t + F(1.0)), op):
        return -1, F(np.inf), np.zeros(6, F), False
    return int(perm[acc_j]), F(out[0]), out[1:7].copy(), sum(t == acc_t for t in ts) > 1


# ============================================================================================ CPU: the oracle's loops
def test_oracle_trace_rays_equals_oracle_render(oracle):
    """Tracing the 200^2 camera rays and packing them gives the reference's frame (oracle_render) bit for bit."""
    h = w = 200
    for name in ("rgbbox", "irreg"):
        pr = oracle.Scene.named(name).prepare(h, w)
        want, rgb, _ = pr.render(h, w, want_rgb=True)
        colour = Q.trace_rays(pr, camera_rays(pr.dump()["cam"], h, w))
        np.testing.assert_array_equal(pack(colour).reshape(h, w), want, err_msg=name)
        np.testing.assert_array_equal(colour.reshape(h, w, 3), rgb, err_msg=name)


@pytest.mark.parametrize("name", ["rgbbox", "random"])
def test_oracle_intersect_rays_equals_brute_force(oracle, name):
    """The oracle's intersect loop (the BVH walk) == a brute-force closest-hit search over all spheres, including rgbbox's
    coincident spheres (tie -> lowest Morton-sorted leaf) and origins inside a sphere."""
    sc = oracle.Scene.rgbbox() if name == "rgbbox" else oracle.Scene.random(300, seed=5)
    spheres, _ = sc.arrays()
    pr = sc.prepare(100, 100)
    perm = pr.dump()["perm"]
    rays = seeded_rays(spheres, 300, seed=11)
    if name == "rgbbox":   # aim at the wall corners, where two walls put a sphere at the same place
        pos = spheres[:, 0:3]
        _, first, counts = np.unique(pos, axis=0, return_index=True, return_counts=True)
        twins = pos[first[counts > 1]]
        assert len(twins) > 0
        k = np.arange(0, 60)
        rays[k, 0:3] = F([0.0, 30.0, 30.0])
        rays[k, 3:6] = twins[k % len(twins)] - rays[k, 0:3]
    index, t, pn = Q.intersect_rays(pr, rays, want_pn=True, threads=4)
    ties = inside = 0
    for k in range(len(rays)):
        bi, bt, bpn, tied = brute_force_objs_hit(oracle, perm, spheres, rays[k])
        assert (index[k], t[k]) == (bi, bt), (k, rays[k], index[k], t[k], bi, bt)
        np.testing.assert_array_equal(pn[k], bpn, err_msg=str(k))
        ties += tied
        if bi >= 0:
            inside += float(np.sum((rays[k, 0:3] - spheres[bi, 0:3]) ** 2)) < float(spheres[bi, 6]) ** 2
    assert (index >= 0).sum() > 50 and (index < 0).sum() > 20
    assert inside > 10
    if name == "rgbbox":
        assert ties > 10


def test_oracle_ray_loops_are_thread_count_independent(oracle):
    pr = oracle.Scene.irreg().prepare(64, 64)
    spheres, _ = oracle.Scene.irreg().arrays()
    rays = seeded_rays(spheres, 2000, seed=3)
    a = Q.intersect_rays(pr, rays, want_pn=True, threads=1)
    b = Q.intersect_rays(pr, rays, want_pn=True, threads=7)
    for x, y in zip(a, b):
        np.testing.assert_array_equal(x, y)
    np.testing.assert_array_equal(Q.trace_rays(pr, rays, threads=1), Q.trace_rays(pr, rays, threads=5))


def test_python_rejects_bad_ray_arrays(R):
    for bad in (np.zeros((4, 5), F), np.zeros((4, 6), np.float64), np.zeros(6, F), [[0.0] * 6]):
        with pytest.raises(R.RayError):
            R.Context._rays(bad)


# ============================================================================================ GPU
def _scene(ctx, name, h=500, w=500):
    if name.startswith("random"):
        n = int(name[len("random"):])
        sc = ctx.scene_random(n, 1)
    else:
        sc = ctx.scene(name)
    return sc, ctx.prepare_scene(h, w, sc)


def _oracle_prepared(oracle, name, h=500, w=500):
    if name.startswith("random"):
        return oracle.Scene.random(int(name[len("random"):]), seed=1).prepare(h, w)
    return oracle.Scene.named(name).prepare(h, w)


def _assert_same_floats(got, want, what):
    # exact, with NaN equal to NaN (degenerate rays)
    np.testing.assert_array_equal(got, want, err_msg=what)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["rgbbox", "irreg"])
def test_trace_camera_rays_equals_golden_png(R, golden, name):
    want, _ = golden[f"{name}_500"]
    with R.Context() as ctx:
        sc, pr = _scene(ctx, name)
        rays = camera_rays(pr.info()["camera"], 500, 500)
        got = pack(ctx.trace(pr, rays)).reshape(500, 500)
        assert int((got != want).sum()) == 0, name


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["rgbbox", "irreg"])
def test_trace_sample_rays_equals_spp4_render(R, name):
    """Every sample ray of a 1000^2 4-spp frame traced, summed in sample order in f32 and scaled by 1/spp == the
    renderer's float framebuffer and pixels, bit for bit."""
    h = w = 1000
    spp = 4
    with R.Context() as ctx:
        sc, pr = _scene(ctx, name, h, w)
        cam = pr.info()["camera"]
        offs = R.host_sample_offsets(spp)
        total = None
        for s in range(spp):
            c = ctx.trace(pr, camera_rays(cam, h, w, offs[s]))
            total = c if s == 0 else total + c
        col = (F(1.0) / F(spp)) * total
        pix, rgb = ctx.render_host(h, w, pr, spp=spp, want_rgb=True)
    np.testing.assert_array_equal(col.reshape(h, w, 3), rgb)
    np.testing.assert_array_equal(pack(col).reshape(h, w), pix)


def _degenerate(rays):
    d = rays.copy()
    d[0, 3:6] = 0.0                       # zero direction
    d[1, 3] = np.inf
    d[2, 0] = np.nan
    d[3, 4] = np.nan
    d[4, 0:3] = -np.inf
    d[5, 3:6] = [np.inf, -np.inf, 0.0]
    return d


@pytest.mark.gpu
@pytest.mark.parametrize("name,n", [("rgbbox", 1), ("rgbbox", 31), ("rgbbox", 33), ("rgbbox", 5000), ("rgbbox", (1 << 20) + 7),
                                    ("irreg", 33), ("irreg", 20000), ("random100000", 20000), ("random1000000", 1 << 16)])
def test_queries_equal_oracle_on_seeded_rays(R, oracle, name, n):
    opr = _oracle_prepared(oracle, name)
    with R.Context() as ctx:
        sc, pr = _scene(ctx, name)
        spheres = sc.arrays()[0]
        rays = seeded_rays(spheres, n, seed=n)
        if n >= 8:
            rays = _degenerate(rays)
        index, t, pn = ctx.intersect(pr, rays, want_pn=True)
        colour = ctx.trace(pr, rays)
    wi, wt, wpn = Q.intersect_rays(opr, rays, want_pn=True)
    np.testing.assert_array_equal(index, wi, err_msg=f"{name} index")
    _assert_same_floats(t, wt, f"{name} t")
    _assert_same_floats(pn, wpn, f"{name} pn")
    _assert_same_floats(colour, Q.trace_rays(opr, rays), f"{name} colour")
    if n >= 1000:
        assert (index >= 0).any() and (index < 0).any()


@pytest.mark.gpu
def test_intersect_device_and_host_built_scenes_and_repeat_runs(R, oracle):
    import torch
    n = 50000
    with R.Context() as ctx, R.Context(host_build=1) as ctx_h:
        for name in ("irreg", "random100000"):
            sc, pr = _scene(ctx, name)
            sc_h, pr_h = _scene(ctx_h, name)
            rays = seeded_rays(sc.arrays()[0], n, seed=7)
            a = ctx.intersect(pr, rays)
            b = ctx_h.intersect(pr_h, rays)
            np.testing.assert_array_equal(a[0], b[0], err_msg=name)
            np.testing.assert_array_equal(a[1], b[1], err_msg=name)
            # device pointers, twice: identical
            dr = torch.from_numpy(rays).cuda()
            outs = []
            for _ in range(2):
                idx = torch.full((n,), -7, dtype=torch.int32, device="cuda")
                t = torch.empty(n, dtype=torch.float32, device="cuda")
                col = torch.empty((n, 3), dtype=torch.float32, device="cuda")
                torch.cuda.synchronize()
                ctx.intersect_into(dr.data_ptr(), n, pr, idx.data_ptr(), t.data_ptr())
                ctx.trace_into(dr.data_ptr(), n, pr, col.data_ptr())
                ctx.sync()
                outs.append((idx.cpu().numpy(), t.cpu().numpy(), col.cpu().numpy()))
            for x, y in zip(outs[0], outs[1]):
                np.testing.assert_array_equal(x, y)
            np.testing.assert_array_equal(outs[0][0], a[0])
            np.testing.assert_array_equal(outs[0][1], a[1])


@pytest.mark.gpu
def test_scene_freed_right_after_async_query(R, oracle):
    """The query reads the scene until it ends: freeing the prepared scene (and preparing others into the freed memory)
    right after the asynchronous call must not change its results."""
    import torch
    n = 1 << 18
    opr = _oracle_prepared(oracle, "irreg")
    with R.Context() as ctx:
        sc, pr = _scene(ctx, "irreg")
        rays = seeded_rays(sc.arrays()[0], n, seed=9)
        dr = torch.from_numpy(rays).cuda()
        idx = torch.empty(n, dtype=torch.int32, device="cuda")
        t = torch.empty(n, dtype=torch.float32, device="cuda")
        col = torch.empty((n, 3), dtype=torch.float32, device="cuda")
        torch.cuda.synchronize()
        ctx.intersect_into(dr.data_ptr(), n, pr, idx.data_ptr(), t.data_ptr())
        ctx.trace_into(dr.data_ptr(), n, pr, col.data_ptr())
        pr.free()
        others = [ctx.prepare_scene(500, 500, ctx.scene_random(20000, s)) for s in range(3)]
        ctx.sync()
        wi, wt, _ = Q.intersect_rays(opr, rays)
        np.testing.assert_array_equal(idx.cpu().numpy(), wi)
        np.testing.assert_array_equal(t.cpu().numpy(), wt)
        np.testing.assert_array_equal(col.cpu().numpy(), Q.trace_rays(opr, rays))
        for o in others:
            o.free()


@pytest.mark.gpu
def test_bad_arguments_launch_nothing(R):
    import torch
    with R.Context() as ctx:
        sc, pr = _scene(ctx, "rgbbox", 64, 64)
        rays = torch.zeros((8, 6), dtype=torch.float32, device="cuda")
        idx = torch.empty(8, dtype=torch.int32, device="cuda")
        t = torch.empty(8, dtype=torch.float32, device="cuda")
        ctx.sync()
        before = ctx.launch_count()
        L, h = ctx.lib, ctx.handle
        bad = [
            L.ray_b200_intersect_into(h, pr.handle, rays.data_ptr(), -1, idx.data_ptr(), t.data_ptr(), None),
            L.ray_b200_intersect_into(h, pr.handle, rays.data_ptr(), (1 << 30) + 1, idx.data_ptr(), t.data_ptr(), None),
            L.ray_b200_intersect_into(h, pr.handle, None, 8, idx.data_ptr(), t.data_ptr(), None),
            L.ray_b200_intersect_into(h, pr.handle, rays.data_ptr(), 8, None, t.data_ptr(), None),
            L.ray_b200_intersect_into(h, pr.handle, rays.data_ptr(), 8, idx.data_ptr(), None, None),
            L.ray_b200_intersect_into(h, None, rays.data_ptr(), 8, idx.data_ptr(), t.data_ptr(), None),
            L.ray_b200_trace_into(h, pr.handle, rays.data_ptr(), 8, None),
            L.ray_b200_trace_into(h, None, rays.data_ptr(), 8, t.data_ptr()),
            L.ray_b200_trace_into(h, pr.handle, rays.data_ptr(), -5, t.data_ptr()),
            L.ray_b200_intersect_host(h, pr.handle, None, 8, np.empty(8, np.int32).ctypes.data, np.empty(8, F).ctypes.data, None),
            L.ray_b200_trace_host(h, pr.handle, np.zeros((8, 6), F).ctypes.data, 8, None),
        ]
        assert all(rc != 0 for rc in bad), bad
        assert ctx.get_error()
        # n = 0: success, nothing launched, null pointers allowed
        assert L.ray_b200_intersect_into(h, pr.handle, None, 0, None, None, None) == 0
        assert L.ray_b200_trace_into(h, pr.handle, None, 0, None) == 0
        empty = ctx.intersect(pr, np.zeros((0, 6), F))
        assert empty[0].shape == (0,) and ctx.trace(pr, np.zeros((0, 6), F)).shape == (0, 3)
        assert ctx.launch_count() == before
        ctx.intersect(pr, np.zeros((8, 6), F))
        assert ctx.launch_count() == before + 1


def _device_count():
    try:
        import torch
        return torch.cuda.device_count()
    except Exception:
        return 0


@pytest.mark.gpu
@pytest.mark.skipif(_device_count() < 2, reason="needs at least 2 GPUs in this process")
def test_multi_gpu_context_refuses_ray_queries(R):
    with R.Context(gpus=2) as ctx:
        sc, pr = _scene(ctx, "rgbbox", 64, 64)
        before = ctx.launch_count()
        with pytest.raises(R.RayError, match="multi-GPU"):
            ctx.intersect(pr, np.zeros((8, 6), F))
        with pytest.raises(R.RayError, match="multi-GPU"):
            ctx.trace(pr, np.zeros((8, 6), F))
        assert ctx.launch_count() == before
