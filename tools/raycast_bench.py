"""Ray-query benchmark (include/ray_b200.h "ray queries"), one JSON document on stdout (and --out).

trace:     the 1000^2 1-spp camera rays of rgbbox and irreg, row-major and in 8x4-tile order (the renderer's tile layout),
           against render_into of the same frame at spp = 1 - the three arms alternated window by window.
intersect: 2^22 seeded rays per scene (rgbbox, irreg, 1 M random spheres), index + t and index + t + pn alternated;
           Mrays/s and the share of the instruction-issue bound of DESIGN.md section 7 (useful thread-instructions of the
           reference traversal's box / sphere tests over SMs x 4 x 32 x SM clock), the work counted on a seeded subsample.

Timing: CUDA events around back-to-back launches on the context's stream, windows of at least --window seconds after a
warm-up, median of --reps windows per arm.  Usage: python tools/raycast_bench.py [--out profiles/r3_raycast.json]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
F = np.float32
MIN_BOX_INSTR, MIN_SPHERE_INSTR = 23, 30   # bench.py's useful-instruction model


def camera_rays(cam12, h, w):
    c = np.asarray(cam12, F)
    u = np.broadcast_to(np.arange(w, dtype=F)[None, :] / F(w), (h, w))
    v = np.broadcast_to((F(h) - np.arange(h, dtype=F))[:, None] / F(h), (h, w))
    rays = np.empty((h, w, 6), F)
    rays[..., 0:3] = c[0:3]
    for k in range(3):
        rays[..., 3 + k] = ((c[3 + k] + u * c[6 + k]) + v * c[9 + k]) - c[k]
    return rays


def tile_order(rays_hw6):
    h, w = rays_hw6.shape[:2]
    assert h % 4 == 0 and w % 8 == 0
    return np.ascontiguousarray(rays_hw6.reshape(h // 4, 4, w // 8, 8, 6).transpose(0, 2, 1, 3, 4).reshape(-1, 6))


def seeded_rays(spheres, n, seed):
    """Half aimed at sphere centres from around the scene, half in random directions (many miss the root box)."""
    rng = np.random.default_rng(seed)
    pos, rad = spheres[:, 0:3], spheres[:, 6]
    lo, hi = pos.min(0) - 2 * rad.max(), pos.max(0) + 2 * rad.max()
    org = lo + rng.random((n, 3), dtype=F) * (hi - lo) * 3 - (hi - lo)
    tgt = pos[rng.integers(0, len(pos), n)]
    d = np.where((rng.random(n) < 0.5)[:, None], tgt - org, rng.standard_normal((n, 3), dtype=F))
    return np.ascontiguousarray(np.concatenate([org, d], 1), F)


def work_counts(packed, root_box, rays):
    """Box and sphere tests of the reference traversal (objs_hit: every inner node whose ancestors' boxes all pass gets a
    box test, every leaf whose parent's box passes a sphere test) for `rays`, walked level by level on the BVH2C arrays
    with the kernels' f32 box test."""
    nodes = packed["nodes"].reshape(-1, 16)
    o, d = rays[:, 0:3].astype(F), rays[:, 3:6].astype(F)
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        inv = F(1.0) / d

        def hit(ray, lo, hi):
            t0, t1 = (lo - o[ray]) * inv[ray], (hi - o[ray]) * inv[ray]
            neg = inv[ray] < 0
            a, b = np.where(neg, t1, t0), np.where(neg, t0, t1)
            tmin = np.fmax(np.fmax(np.fmax(a[:, 0], F(0)), a[:, 1]), a[:, 2])
            tmax = np.fmin(np.fmin(np.fmin(b[:, 0], F(1e9)), b[:, 1]), b[:, 2])
            return ~(tmax <= tmin)

        ray = np.arange(len(rays))
        box_tests, leaf_tests = len(rays), 0
        rb = np.asarray(root_box, F)
        ray = ray[hit(ray, rb[None, 0:3], rb[None, 3:6])]
        node = np.zeros(len(ray), np.int64)
        while len(ray):
            q = nodes[node]
            lptr, rptr = q[:, 3].view(np.int32), q[:, 7].view(np.int32)
            nxt_r, nxt_n = [], []
            for ptr, lo, hi in ((lptr, q[:, 0:3], q[:, 4:7]), (rptr, q[:, 8:11], q[:, 12:15])):
                leaf = ptr < 0
                leaf_tests += int(leaf.sum())
                box_tests += int((~leaf).sum())
                k = ~leaf & hit(ray, lo, hi)
                nxt_r.append(ray[k])
                nxt_n.append(ptr[k].astype(np.int64))
            ray, node = np.concatenate(nxt_r), np.concatenate(nxt_n)
    return box_tests, leaf_tests


def nvsmi(fields):
    try:
        out = subprocess.run(["nvidia-smi", "--id=0", f"--query-gpu={fields}", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=20).stdout.strip()
        return [x.strip() for x in out.split(",")]
    except Exception:
        return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--window", type=float, default=1.0, help="seconds per timed window")
    ap.add_argument("--reps", type=int, default=3, help="timed windows per arm")
    ap.add_argument("--n-intersect", type=int, default=1 << 22)
    args = ap.parse_args()

    import torch
    import raytracers_b200 as R

    res = {"device": torch.cuda.get_device_name(0), "window_s": args.window, "reps": args.reps}
    pw = nvsmi("power.limit,power.default_limit,clocks.max.sm")
    if pw:
        res["power_limit_w"], res["power_default_limit_w"], res["sm_max_mhz"] = pw
    ctx = R.Context(device=0)
    sm_count = torch.cuda.get_device_properties(0).multi_processor_count
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def window(fn):
        """ms per call: back-to-back calls until one timed batch lasts >= args.window seconds."""
        k = 1
        while True:
            ctx.sync()
            torch.cuda.synchronize()
            ev0.record(torch.cuda.current_stream())
            for _ in range(k):
                fn()
            ev1.record(torch.cuda.current_stream())
            ev1.synchronize()
            ms = ev0.elapsed_time(ev1)
            if ms >= 1000.0 * args.window:
                return ms / k
            k = max(k * 2, int(k * 1.2 * 1000.0 * args.window / max(ms, 1e-3)))

    def alternate(arms):
        for fn in arms.values():   # warm-up (module load, shared-memory opt-in, clocks)
            for _ in range(20):
                fn()
        times = {a: [] for a in arms}
        for _ in range(args.reps):
            for a, fn in arms.items():
                times[a].append(window(fn))
        return {a: {"ms_median": float(np.median(v)), "ms": [round(x, 5) for x in v]} for a, v in times.items()}

    ctx.set_stream(torch.cuda.current_stream().cuda_stream)
    # ---------------------------------------------------------------- trace vs render, 1000^2 1 spp
    h = w = 1000
    res["trace"] = {}
    for name in ("rgbbox", "irreg"):
        sc = ctx.scene(name)
        pr = ctx.prepare_scene(h, w, sc)
        rays = camera_rays(pr.info()["camera"], h, w)
        row = torch.from_numpy(np.ascontiguousarray(rays.reshape(-1, 6))).cuda()
        tile = torch.from_numpy(tile_order(rays)).cuda()
        col = torch.empty((h * w, 3), dtype=torch.float32, device="cuda")
        pix = torch.empty((h, w), dtype=torch.int32, device="cuda")
        rgb = torch.empty((h, w, 3), dtype=torch.float32, device="cuda")
        # the traced colours are the render's float framebuffer
        ctx.render_into(pix.data_ptr(), h, w, pr, spp=1, out_rgb_dev=rgb.data_ptr())
        ctx.trace_into(row.data_ptr(), h * w, pr, col.data_ptr())
        torch.cuda.synchronize()
        same = bool(torch.equal(col.view(h, w, 3), rgb))
        arms = {"render_into_spp1": lambda: ctx.render_into(pix.data_ptr(), h, w, pr, spp=1),
                "trace_row_major": lambda: ctx.trace_into(row.data_ptr(), h * w, pr, col.data_ptr()),
                "trace_tile_order": lambda: ctx.trace_into(tile.data_ptr(), h * w, pr, col.data_ptr())}
        r = alternate(arms)
        base = r["render_into_spp1"]["ms_median"]
        for a in ("trace_row_major", "trace_tile_order"):
            r[a]["vs_render"] = round(r[a]["ms_median"] / base, 3)
            r[a]["mrays_per_s"] = round(h * w / (r[a]["ms_median"] * 1e-3) / 1e6, 1)
        r["colours_equal_render_rgb"] = same
        res["trace"][name] = r
        pr.free(); sc.free()
        print(name, json.dumps(r), file=sys.stderr, flush=True)

    # ---------------------------------------------------------------- intersect, 2^22 seeded rays
    n = args.n_intersect
    res["intersect"] = {}
    for name in ("rgbbox", "irreg", "random1000000"):
        sc = ctx.scene_random(1000000, 1) if name.startswith("random") else ctx.scene(name)
        pr = ctx.prepare_scene(h, w, sc)
        spheres = sc.arrays()[0]
        rays_np = seeded_rays(spheres, n, seed=2024)
        rays = torch.from_numpy(rays_np).cuda()
        idx = torch.empty(n, dtype=torch.int32, device="cuda")
        t = torch.empty(n, dtype=torch.float32, device="cuda")
        pn = torch.empty((n, 6), dtype=torch.float32, device="cuda")
        arms = {"index_t": lambda: ctx.intersect_into(rays.data_ptr(), n, pr, idx.data_ptr(), t.data_ptr()),
                "index_t_pn": lambda: ctx.intersect_into(rays.data_ptr(), n, pr, idx.data_ptr(), t.data_ptr(), pn.data_ptr())}
        r = alternate(arms)
        clk = nvsmi("clocks.sm")
        sm_mhz = float(clk[0]) if clk and clk[0].replace(".", "").isdigit() else 1965.0
        sub = rays_np[np.random.default_rng(1).choice(n, 1 << 16, replace=False)]
        for a in arms:
            r[a]["mrays_per_s"] = round(n / (r[a]["ms_median"] * 1e-3) / 1e6, 1)
        try:
            boxes, leaves = work_counts(pr.packed(), pr.info()["root_box"], sub)
            useful = (MIN_BOX_INSTR * boxes + MIN_SPHERE_INSTR * leaves) * (n / len(sub))
            for a in arms:
                r[a]["issue_frac"] = round(useful / (r[a]["ms_median"] * 1e-3) / (sm_count * 4 * 32 * sm_mhz * 1e6), 4)
            r["work_per_ray"] = {"box_tests": round(boxes / len(sub), 2), "leaf_tests": round(leaves / len(sub), 2),
                                 "counted_on": len(sub)}
        except Exception as e:  # the timings stand without the work count
            r["work_per_ray"] = {"error": repr(e)}
        r["hit_fraction"] = round(float((idx.cpu().numpy() >= 0).mean()), 4)
        r["sm_mhz_after"] = sm_mhz
        res["intersect"][name] = r
        pr.free(); sc.free()
        print(name, json.dumps(r), file=sys.stderr, flush=True)
    ctx.close()
    res["library_bytes"] = os.path.getsize(R.lib_path())
    js = json.dumps(res, indent=1)
    print(js)
    if args.out:
        with open(args.out, "w") as f:
            f.write(js + "\n")


if __name__ == "__main__":
    main()
