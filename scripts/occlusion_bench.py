"""Occlusion queries (rt_occluded_rays_device) on one GPU, against the closest-hit ray query (rt_trace_rays_device with
only the prim output) on the same ray buffers.

    python scripts/occlusion_bench.py [--reps 20] [--width 3840 --height 2160] [--worlds c3,c5] [--out DIR]

For each world the first-hit buffers of a fixed-jitter W x H frame (render_aov_device) give the hit pixels' positions.
Four workloads of rays, each packed once on the device:
  shadow     from every hit pixel's first-hit position towards a point light above the world's bounds (every
             sphere's centre +- radius, every triangle vertex): centred in x and z, 10 units above their
             top; t_max = |L - p|
  camera     the un-normalised camera vector of every pixel centre (scripts/rays_bench.py camera_rays), t_max = +inf
  incoherent W*H rays from first-hit positions (drawn with replacement) in uniformly random directions, t_max = +inf
  all_miss   W*H rays from the light's position in random directions of the upper cone d.y > 0.5 |d|, away from the
             whole world, t_max = +inf; the run stops unless every one of them is answered 0
The answers are first checked to agree for every ray (occluded == (prim >= 0 ? 1 : prim == -1 ? 0 : 2)).  The two calls
then alternate, --reps times each, with the L2 flushed (256 MiB write) between calls; kernel times come from the
library's CUDA events (RenderStats.kernel_ms).  Reports the occluded fraction, the medians and the ratio of the medians
(occlusion / closest hit), with and without RT_OPT_GROUP_CULL for worlds where it applies.  The card's name and power
limit are read in the same run.  Prints one JSON line; --out DIR also writes it to DIR/occlusion_bench.json.
"""
from __future__ import annotations

import argparse
import importlib
import json
import statistics
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "scripts"))
from rays_bench import camera_rays, card  # noqa: E402


def scene_bounds(h):
    """The world's bounds: every sphere's centre +- |radius| and every triangle vertex (float64 lo[3], hi[3])."""
    pts = []
    for i in range(h.n_spheres):
        s = h.sphere(i).astype(np.float64)
        pts += [s[0:3] - abs(s[3]), s[0:3] + abs(s[3])]
    for j in range(h.n_triangles):
        t = h.triangle(j).astype(np.float64)
        pts += [t[0:3], t[3:6], t[6:9]]
    pts = np.array(pts)
    return pts.min(0), pts.max(0)


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--width", type=int, default=3840)
    ap.add_argument("--height", type=int, default=2160)
    ap.add_argument("--worlds", default="c3,c5")
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    import torch
    rt = importlib.import_module("rust-swift-raytracer_b200")
    scenes = importlib.import_module("rust-swift-raytracer_b200.scenes")
    if rt.device_count() < 1:
        raise SystemExit("occlusion_bench needs a CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    W, H = a.width, a.height
    N = W * H
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)        # > 126 MB L2
    g = torch.Generator(device=dev).manual_seed(4321)
    result = {"card": card(), "width": W, "height": H, "reps": a.reps,
              "l2": "flushed between calls (256 MiB write)", "worlds": {}}

    def pack(o, d, t_max):
        n = d.shape[0]
        r = torch.zeros((n, 8), dtype=torch.float32, device=dev)
        r[:, 0:3] = o
        r[:, 3] = t_max
        r[:, 4:7] = d
        return r

    def unit(n):
        d = torch.randn((n, 3), device=dev, generator=g)
        return d / d.norm(dim=1, keepdim=True)

    for key in a.worlds.split(","):
        h = rt.load_world(getattr(scenes, key + "_world")())
        aov = rt.render_aov(h, W, H, rt.Options(fixed_jitter=True, device=0))
        pos = aov["position"][aov["prim"] >= 0].reshape(-1, 3).contiguous()
        lo, hi = scene_bounds(h)
        light = torch.tensor([(lo[0] + hi[0]) / 2, hi[1] + 10.0, (lo[2] + hi[2]) / 2],
                             dtype=torch.float32, device=dev)
        cam_rays, _ = camera_rays(h.camera_floats(), W, H)
        idx = torch.randint(0, pos.shape[0], (N,), device=dev, generator=g)
        up = unit(4 * N)
        up = up[up[:, 1] > 0.5][:N]
        to_l = light[None, :] - pos
        workloads = {
            "shadow": pack(pos, to_l, to_l.norm(dim=1)),
            "camera": torch.from_numpy(cam_rays).to(dev),
            "incoherent": pack(pos[idx], unit(N), float("inf")),
            "all_miss": pack(light.expand(up.shape[0], 3), up, float("inf")),
        }
        del up, idx, to_l
        occ = torch.empty(N, dtype=torch.uint8, device=dev)                # every workload has at most N rays
        prim = torch.empty(N, dtype=torch.int32, device=dev)
        torch.cuda.synchronize()      # packed on torch's stream; the calls below run on the library's
        rw = {}
        for cull in (False, True):
            q = rt.RayQueryOptions(group_cull=cull, device=0)
            for name, rays in workloads.items():
                n = rays.shape[0]
                st = rt.RenderStats()
                for _ in range(3):                                     # warm-up: modules, scene upload, occupancy
                    rt.occluded_rays_device(h, q, n, rays.data_ptr(), occ.data_ptr(), stats=st)
                    rt.trace_rays_device(h, q, n, rays.data_ptr(), prim=prim.data_ptr(), stats=st)
                p = prim[:n]
                want = torch.where(p >= 0, 1, torch.where(p == -1, 0, 2)).to(torch.uint8)
                agree = bool(torch.equal(occ[:n], want))
                if not agree:
                    raise SystemExit(f"{key}/{name}/cull={cull}: occluded_rays disagrees with trace_rays' prim on "
                                     f"{int((occ[:n] != want).sum())} of {n} rays")
                if name == "all_miss" and bool((occ[:n] != 0).any()):
                    raise SystemExit(f"{key}: {int((occ[:n] != 0).sum())} all-miss rays are not answered 0")
                t_occ, t_hit = [], []
                for _ in range(a.reps):
                    flush.zero_(); torch.cuda.synchronize()
                    rt.occluded_rays_device(h, q, n, rays.data_ptr(), occ.data_ptr(), stats=st)
                    t_occ.append(st.kernel_ms)
                    geo = {k: getattr(st, k) for k in ("grid", "block", "resident", "smem_bytes", "filtered", "culled")}
                    flush.zero_(); torch.cuda.synchronize()
                    rt.trace_rays_device(h, q, n, rays.data_ptr(), prim=prim.data_ptr(), stats=st)
                    t_hit.append(st.kernel_ms)
                mo, mh = statistics.median(t_occ), statistics.median(t_hit)
                rw[f"{name}{'_cull' if cull else ''}"] = {
                    "rays": n, "answers_agree": agree, "occluded_fraction": float((occ[:n] == 1).float().mean()),
                    "occluded_kernel_ms": {"median": mo, "min": min(t_occ), "max": max(t_occ)},
                    "trace_prim_kernel_ms": {"median": mh, "min": min(t_hit), "max": max(t_hit)},
                    "ratio_of_medians": mo / mh, "launch": geo}
        result["worlds"][key] = {"hit_pixels": int(pos.shape[0]), "light": [float(x) for x in light], "workloads": rw}
        del workloads, occ, prim, pos, aov
        torch.cuda.empty_cache()
    line = json.dumps(result)
    print(line, flush=True)
    if a.out:
        Path(a.out).mkdir(parents=True, exist_ok=True)
        (Path(a.out) / "occlusion_bench.json").write_text(line + "\n")


if __name__ == "__main__":
    main()
