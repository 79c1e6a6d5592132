"""The variant matrix: every instantiated render, first-hit, ray-query and occlusion kernel against its reference.

The library never runs "the render kernel"; it runs one of 102 template instantiations that choose_variant /
choose_aov_variant (csrc/rt_kernels.cuh) pick from the world's shape — the walk (DIRECT below 64 spheres, FILTER from
64, CULL on request), where the hot lists live (shared memory with 256-thread CTAs up to 56 KB, 1024-thread CTAs up to
smem_optin - 1024, global memory above), whether the world has triangles, and RT_PATHS_PER_LANE.  The instantiations
differ in register caps, spills, staging and CTA width, so each one is a kernel of its own to test.

MATRIX below has one row per instantiation, keyed by kernel and template arguments: either the worlds that select it
(with the options), or why no world can.  `choose` is a plain restatement of the geometry choice — a test oracle like
the CPU oracle, not product code.  CPU tests: the rows are exactly the instantiations in the built objects, the
restatement picks each "run" row's instantiation for its worlds on a B200 (232,448 bytes of opt-in shared memory), and
the "unreachable" rows are unreachable.  GPU tests (`-m gpu`), one case per "run" row: the launch statistics first
(a world that lands on another instantiation fails, it does not pass against the wrong kernel), then

  * exact render: RGBA8, ray count and the float4 colour sums bit for bit against the oracle (ob.ray_trace);
  * fast-math render: the bars of test_gpu_parity's fast-math test against the exact kernel on the same world, and
    fast CULL == fast FILTER bit for bit on every world of at least 64 spheres;
  * first-hit, ray-query and occlusion kernels: bit for bit against test_aov / test_rays / test_occlusion's references.

The two-paths-per-lane rows run in one subprocess (RT_PATHS_PER_LANE is read once per process).  test_switch_points
puts worlds on the switch points of choose_variant: hot lists of exactly 57,344 bytes and the next size up, exactly the
staging limit and the next size up, solved from the device's own opt-in shared memory.
"""
from __future__ import annotations

import json
import os
import re
import shutil
import subprocess
import sys
import zlib
from pathlib import Path
from typing import NamedTuple

import numpy as np
import pytest

import cases
import test_aov
import test_occlusion
import test_rays

ROOT = Path(__file__).resolve().parent.parent
OBJ = ROOT / "rust-swift-raytracer_b200" / "lib" / "obj"

DIRECT, FILTER, CULL = 0, 1, 2                      # RT_SPH_* of rt_types.h
WALKS = {"DIRECT": DIRECT, "FILTER": FILTER, "CULL": CULL}
WALK_NAMES = {v: k for k, v in WALKS.items()}
FILTER_FROM = 64                                    # RT_FILTER_FROM
LARGE_SMEM_FROM = 56 * 1024                         # kLargeSmemFrom
B200_SMEM_OPTIN = 232448                            # cudaDevAttrMaxSharedMemoryPerBlockOptin of a B200


# ------------------------------------------------------------------------------------- restatement of the choice

def _up(n: int, k: int) -> int:
    return -(-n // k) * k


class Counts(NamedTuple):
    n_sph: int
    n_sph_pad: int
    n_tri_pad: int
    n_groups: int


def packed_counts(radii, n_tri: int) -> Counts:
    """World::packed's list sizes: spheres padded to 8, triangles to 2; from 64 spheres, the cull groups — spheres of
    radius above 8x the median (or not finite) in groups of 8 that always pass, the rest in groups of 8, the count rounded
    up to 32 (rt_scene.cpp cull_order)."""
    r = np.abs(np.asarray(radii, np.float32))
    S = len(r)
    groups = 0
    if S >= FILTER_FROM:
        big = np.float32(8.0) * np.partition(r, S // 2)[S // 2]
        large = int(np.count_nonzero(~(r <= big)))
        groups = _up(-(-large // 8) + -(-(S - large) // 8), 32)
    return Counts(S, _up(S, 8), _up(int(n_tri), 2), groups)


def hot_bytes(c: Counts, walk: int) -> int:
    """rt_hot_bytes: block C {cull_bound | cull_sph | tri_plane}, block B {sph_filter | tri_plane | sph_r2} or block A."""
    if walk == CULL:
        return (10 * c.n_groups + c.n_tri_pad) * 16
    b = (c.n_sph_pad + c.n_tri_pad) * 16
    if walk == FILTER:
        b += _up(c.n_sph_pad * 4, 16)
    return b


class Variant(NamedTuple):
    smem: bool
    block: int
    walk: int
    tris: bool
    hot: int
    np: int


def choose(c: Counts, cull: bool, paths_per_lane: int, smem_optin: int, lane_kernel: bool = False) -> Variant:
    """choose_variant (render) or choose_aov_variant (lane_kernel: the first-hit, ray and occlusion kernels)."""
    smem_limit = smem_optin - 1024 if smem_optin > 1024 else 0
    walk = CULL if (cull and c.n_groups > 0) else FILTER if c.n_sph >= FILTER_FROM else DIRECT
    hot = hot_bytes(c, walk)
    smem = hot <= smem_limit
    np_ = paths_per_lane if (walk == FILTER and not lane_kernel) else 1
    block = (512 if np_ == 2 else 1024) if (smem and hot > LARGE_SMEM_FROM) else 256
    return Variant(smem, block, walk, c.n_tri_pad > 0, hot, np_)


# ------------------------------------------------------------------------------------------------ row keys

KERNELS = ("render-exact", "render-fast", "aov", "ray", "occlusion")
ID = re.compile(r"^(render-exact|render-fast|aov|ray|occlusion)-(smem|global)(\d+)-(DIRECT|FILTER|CULL)-(tris|notris)(-np2)?$")


class Key(NamedTuple):
    kernel: str
    smem: bool
    block: int
    walk: int
    tris: bool
    np: int


def key_of(row_id: str) -> Key:
    m = ID.match(row_id)
    assert m, f"malformed row id {row_id!r}"
    return Key(m[1], m[2] == "smem", int(m[3]), WALKS[m[4]], m[5] == "tris", 2 if m[6] else 1)


def id_of(k: Key) -> str:
    return (f"{k.kernel}-{'smem' if k.smem else 'global'}{k.block}-{WALK_NAMES[k.walk]}-{'tris' if k.tris else 'notris'}"
            + ("-np2" if k.np == 2 else ""))


def key_for(kernel: str, v: Variant) -> Key:
    return Key(kernel, v.smem, v.block, v.walk, v.tris, v.np)


# ---------------------------------------------------------------------------------------------------- worlds
# name -> (scene text builder, frame (W, H, spp, depth) of the exact render).  S is not a multiple of 8 and T is odd
# wherever the row allows, so that the NaN pads of a partial sphere group, cull group and triangle pair are walked.

BACKDROP = "triangle v0 -40.0 -0.5 -20.0 v1 40.0 -0.5 -20.0 v2 0.0 40.0 -20.0 material GROUND;\n"


def _syn(S, T, seed):
    """scenes.synthetic_world with T triangles, the last of them a backdrop behind the spheres: the triangle next to
    the pad of the last pair is in every frame and in the path of many query rays, so a walk that drops it fails."""
    if T == 0:
        return lambda scenes: scenes.synthetic_world(S, 0, seed=seed)
    return lambda scenes: scenes.synthetic_world(S, T - 1, seed=seed) + BACKDROP


def _rand(seed, S, T):
    return lambda scenes: cases.random_world(seed, S, T)


SMALL, BIG, DEEP = (64, 36, 2, 8), (48, 27, 2, 8), (48, 27, 2, 16)
WORLDS = {
    "default":        (lambda scenes: scenes.default_world(), SMALL),      # 8 spheres
    "example":        (lambda scenes: scenes.example_world(), SMALL),      # 8 spheres + 2 triangles
    "s63":            (_syn(63, 0, 63), SMALL),                            # the last DIRECT world (pads to 64)
    "s64":            (_syn(64, 0, 64), SMALL),                            # the first FILTER world
    "s65":            (_syn(65, 0, 65), SMALL),
    "s801t201":       (_syn(801, 201, 10000), SMALL),                      # c5mini, ragged
    "s4001":          (_syn(4001, 0, 4001), BIG),
    "s8001t2001":     (_syn(8001, 2001, 10000), DEEP),                     # c5, ragged
    "s16001":         (_syn(16001, 0, 4242), BIG),
    "s15001t501":     (_syn(15001, 501, 77), BIG),
    "s37t4001":       (_syn(37, 4001, 37), BIG),                           # a mesh with few spheres
    "s37t15001":      (_syn(37, 15001, 38), BIG),
    # awkward geometry (cases.random_world): needles, degenerate and far triangles, huge spheres ("always" groups)
    "rand45t9":       (_rand(4501, 45, 9), SMALL),
    "rand70":         (_rand(7001, 70, 0), SMALL),
    "rand71t13":      (_rand(7101, 71, 13), SMALL),
    "rand3001t1001":  (_rand(3001, 3001, 1001), BIG),
    "rand16001t1":    (_rand(16001, 16001, 1), BIG),
}


class Run(NamedTuple):
    """A reachable row: the worlds that select it, with group_cull on or off.  fast_math and RT_PATHS_PER_LANE=2
    follow from the key (render-fast, -np2)."""
    worlds: tuple
    cull: bool = False


class Unreachable(NamedTuple):
    reason: str


def run(*worlds, cull=False):
    return Run(tuple(worlds), cull)


DEAD_DIRECT = Unreachable("DIRECT means at most 63 spheres: without triangles at most 64 x 16 = 1,024 hot bytes, "
                          "never above 57,344")

MATRIX = {
    # rt_render_kernel<FAST=false, SMEM, BLOCK, SPH, TRIS, NP=1>
    "render-exact-smem256-DIRECT-notris":     run("default", "s63"),
    "render-exact-smem256-DIRECT-tris":       run("example", "rand45t9"),
    "render-exact-smem1024-DIRECT-notris":    DEAD_DIRECT,
    "render-exact-smem1024-DIRECT-tris":      run("s37t4001"),
    "render-exact-global256-DIRECT-notris":   DEAD_DIRECT,
    "render-exact-global256-DIRECT-tris":     run("s37t15001"),
    "render-exact-smem256-FILTER-notris":     run("s65", "s64", "rand70"),
    "render-exact-smem256-FILTER-tris":       run("s801t201", "rand71t13"),
    "render-exact-smem1024-FILTER-notris":    run("s4001"),
    "render-exact-smem1024-FILTER-tris":      run("s8001t2001", "rand3001t1001"),
    "render-exact-global256-FILTER-notris":   run("s16001"),
    "render-exact-global256-FILTER-tris":     run("s15001t501", "rand16001t1"),
    "render-exact-smem256-CULL-notris":       run("s65", "s64", "rand70", cull=True),
    "render-exact-smem256-CULL-tris":         run("s801t201", "rand71t13", cull=True),
    "render-exact-smem1024-CULL-notris":      run("s4001", cull=True),
    "render-exact-smem1024-CULL-tris":        run("s8001t2001", "rand3001t1001", cull=True),
    "render-exact-global256-CULL-notris":     run("s16001", cull=True),
    "render-exact-global256-CULL-tris":       run("s15001t501", "rand16001t1", cull=True),
    # rt_render_kernel<FAST=false, SMEM, BLOCK, FILTER, TRIS, NP=2>
    "render-exact-smem256-FILTER-notris-np2":  run("s65", "rand70"),
    "render-exact-smem256-FILTER-tris-np2":    run("s801t201", "rand71t13"),
    "render-exact-smem512-FILTER-notris-np2":  run("s4001"),
    "render-exact-smem512-FILTER-tris-np2":    run("s8001t2001", "rand3001t1001"),
    "render-exact-global256-FILTER-notris-np2": run("s16001"),
    "render-exact-global256-FILTER-tris-np2":  run("s15001t501"),
    # rt_render_kernel<FAST=true, SMEM, BLOCK, SPH, TRIS, NP=1> (statistical bars: synthetic worlds)
    "render-fast-smem256-DIRECT-notris":      run("default", "s63"),
    "render-fast-smem256-DIRECT-tris":        run("example"),
    "render-fast-smem1024-DIRECT-notris":     DEAD_DIRECT,
    "render-fast-smem1024-DIRECT-tris":       run("s37t4001"),
    "render-fast-global256-DIRECT-notris":    DEAD_DIRECT,
    "render-fast-global256-DIRECT-tris":      run("s37t15001"),
    "render-fast-smem256-FILTER-notris":      run("s65", "s64"),
    "render-fast-smem256-FILTER-tris":        run("s801t201"),
    "render-fast-smem1024-FILTER-notris":     run("s4001"),
    "render-fast-smem1024-FILTER-tris":       run("s8001t2001"),
    "render-fast-global256-FILTER-notris":    run("s16001"),
    "render-fast-global256-FILTER-tris":      run("s15001t501"),
    "render-fast-smem256-CULL-notris":        run("s65", "s64", cull=True),
    "render-fast-smem256-CULL-tris":          run("s801t201", cull=True),
    "render-fast-smem1024-CULL-notris":       run("s4001", cull=True),
    "render-fast-smem1024-CULL-tris":         run("s8001t2001", cull=True),
    "render-fast-global256-CULL-notris":      run("s16001", cull=True),
    "render-fast-global256-CULL-tris":        run("s15001t501", cull=True),
    # rt_render_kernel<FAST=true, SMEM, BLOCK, FILTER, TRIS, NP=2>
    "render-fast-smem256-FILTER-notris-np2":  run("s65"),
    "render-fast-smem256-FILTER-tris-np2":    run("s801t201"),
    "render-fast-smem512-FILTER-notris-np2":  run("s4001"),
    "render-fast-smem512-FILTER-tris-np2":    run("s8001t2001"),
    "render-fast-global256-FILTER-notris-np2": run("s16001"),
    "render-fast-global256-FILTER-tris-np2":  run("s15001t501"),
    # rt_aov_kernel<SMEM, BLOCK, SPH, TRIS>
    "aov-smem256-DIRECT-notris":              run("default", "s63"),
    "aov-smem256-DIRECT-tris":                run("example", "rand45t9"),
    "aov-smem1024-DIRECT-notris":             DEAD_DIRECT,
    "aov-smem1024-DIRECT-tris":               run("s37t4001"),
    "aov-global256-DIRECT-notris":            DEAD_DIRECT,
    "aov-global256-DIRECT-tris":              run("s37t15001"),
    "aov-smem256-FILTER-notris":              run("s65", "s64", "rand70"),
    "aov-smem256-FILTER-tris":                run("s801t201", "rand71t13"),
    "aov-smem1024-FILTER-notris":             run("s4001"),
    "aov-smem1024-FILTER-tris":               run("s8001t2001", "rand3001t1001"),
    "aov-global256-FILTER-notris":            run("s16001"),
    "aov-global256-FILTER-tris":              run("s15001t501", "rand16001t1"),
    "aov-smem256-CULL-notris":                run("s65", "s64", "rand70", cull=True),
    "aov-smem256-CULL-tris":                  run("s801t201", "rand71t13", cull=True),
    "aov-smem1024-CULL-notris":               run("s4001", cull=True),
    "aov-smem1024-CULL-tris":                 run("s8001t2001", "rand3001t1001", cull=True),
    "aov-global256-CULL-notris":              run("s16001", cull=True),
    "aov-global256-CULL-tris":                run("s15001t501", "rand16001t1", cull=True),
    # rt_ray_kernel<SMEM, BLOCK, SPH, TRIS>
    "ray-smem256-DIRECT-notris":              run("default", "s63"),
    "ray-smem256-DIRECT-tris":                run("example", "rand45t9"),
    "ray-smem1024-DIRECT-notris":             DEAD_DIRECT,
    "ray-smem1024-DIRECT-tris":               run("s37t4001"),
    "ray-global256-DIRECT-notris":            DEAD_DIRECT,
    "ray-global256-DIRECT-tris":              run("s37t15001"),
    "ray-smem256-FILTER-notris":              run("s65", "s64", "rand70"),
    "ray-smem256-FILTER-tris":                run("s801t201", "rand71t13"),
    "ray-smem1024-FILTER-notris":             run("s4001"),
    "ray-smem1024-FILTER-tris":               run("s8001t2001", "rand3001t1001"),
    "ray-global256-FILTER-notris":            run("s16001"),
    "ray-global256-FILTER-tris":              run("s15001t501", "rand16001t1"),
    "ray-smem256-CULL-notris":                run("s65", "s64", "rand70", cull=True),
    "ray-smem256-CULL-tris":                  run("s801t201", "rand71t13", cull=True),
    "ray-smem1024-CULL-notris":               run("s4001", cull=True),
    "ray-smem1024-CULL-tris":                 run("s8001t2001", "rand3001t1001", cull=True),
    "ray-global256-CULL-notris":              run("s16001", cull=True),
    "ray-global256-CULL-tris":                run("s15001t501", "rand16001t1", cull=True),
    # rt_occlusion_kernel<SMEM, BLOCK, SPH, TRIS>
    "occlusion-smem256-DIRECT-notris":        run("default", "s63"),
    "occlusion-smem256-DIRECT-tris":          run("example", "rand45t9"),
    "occlusion-smem1024-DIRECT-notris":       DEAD_DIRECT,
    "occlusion-smem1024-DIRECT-tris":         run("s37t4001"),
    "occlusion-global256-DIRECT-notris":      DEAD_DIRECT,
    "occlusion-global256-DIRECT-tris":        run("s37t15001"),
    "occlusion-smem256-FILTER-notris":        run("s65", "s64", "rand70"),
    "occlusion-smem256-FILTER-tris":          run("s801t201", "rand71t13"),
    "occlusion-smem1024-FILTER-notris":       run("s4001"),
    "occlusion-smem1024-FILTER-tris":         run("s8001t2001", "rand3001t1001"),
    "occlusion-global256-FILTER-notris":      run("s16001"),
    "occlusion-global256-FILTER-tris":        run("s15001t501", "rand16001t1"),
    "occlusion-smem256-CULL-notris":          run("s65", "s64", "rand70", cull=True),
    "occlusion-smem256-CULL-tris":            run("s801t201", "rand71t13", cull=True),
    "occlusion-smem1024-CULL-notris":         run("s4001", cull=True),
    "occlusion-smem1024-CULL-tris":           run("s8001t2001", "rand3001t1001", cull=True),
    "occlusion-global256-CULL-notris":        run("s16001", cull=True),
    "occlusion-global256-CULL-tris":          run("s15001t501", "rand16001t1", cull=True),
}

RUN_ROWS = [r for r, v in MATRIX.items() if isinstance(v, Run)]


def _rows(kernels, np2):
    return [r for r in RUN_ROWS if key_of(r).kernel in kernels and (key_of(r).np == 2) == np2]


# ------------------------------------------------------------------------------------------------ shared state
# World texts, oracle worlds and product handles are built once per process: the big worlds take a second each.

_texts, _oracle_worlds, _handles, _renders = {}, {}, {}, {}


def world_text(scenes, name):
    if name not in _texts:
        _texts[name] = WORLDS[name][0](scenes)
    return _texts[name]


def oracle_world(ob, scenes, name):
    if name not in _oracle_worlds:
        _oracle_worlds[name] = ob.parse_input(world_text(scenes, name))
    return _oracle_worlds[name]


def counts_of(ob, scenes, name) -> Counts:
    _, world = oracle_world(ob, scenes, name)
    return packed_counts([s.radius for s in world.spheres()], world.n_triangles)


def handle(rt, scenes, name):
    if name not in _handles:
        _handles[name] = rt.load_world(world_text(scenes, name))
    return _handles[name]


def oracle_render(ob, scenes, name):
    """(pixels, rays, float4 sums) of the world's exact frame."""
    if name not in _renders:
        cam, world = oracle_world(ob, scenes, name)
        W, H, spp, depth = WORLDS[name][1]
        _renders[name] = ob.ray_trace(world, cam, W, H, spp, depth, want_accum=True)
    return _renders[name]


def smem_optin_of_device() -> int:
    import torch
    return int(torch.cuda.get_device_properties(torch.cuda.current_device()).shared_memory_per_block_optin)


def expected_stats(v: Variant) -> dict:
    return {"block": v.block, "resident": int(v.smem), "smem_bytes": v.hot if v.smem else 0,
            "filtered": int(v.walk != DIRECT), "culled": int(v.walk == CULL), "paths_per_lane": v.np}


def check_stats(where, st, v: Variant):
    want = expected_stats(v)
    got = {k: int(getattr(st, k)) for k in want}
    assert got == want, f"{where}: launch statistics {got}, the restatement predicts {want}"


def selected(ob, scenes, row_id, world, smem_optin) -> Variant:
    """The restatement's variant for the row's world and options; it must be the row's instantiation."""
    k, spec = key_of(row_id), MATRIX[row_id]
    v = choose(counts_of(ob, scenes, world), spec.cull, k.np, smem_optin, lane_kernel=not k.kernel.startswith("render"))
    assert key_for(k.kernel, v) == k, f"{row_id}: world {world} selects {id_of(key_for(k.kernel, v))} on this device"
    return v


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def _rmse(a, b):
    d = a[:, :, :3].astype(np.float64) - b[:, :, :3].astype(np.float64)
    return float(np.sqrt((d * d).mean()))


def _render(rt, h, W, H, spp, depth, **kw):
    fb, st = rt.Framebuffer(W, H), rt.RenderStats()
    rt.render_with_options(fb, h, rt.Options(spp, depth, **kw), st)
    return fb.pixels.copy(), st


# ------------------------------------------------------------------------------------------------ the checks
# Plain functions of (rt, ob, scenes, row, smem_optin): the GPU tests call them, and so does the subprocess of the
# two-paths-per-lane rows.

def check_render_exact(rt, ob, scenes, row, smem_optin):
    import torch
    cull = MATRIX[row].cull
    for name in MATRIX[row].worlds:
        v = selected(ob, scenes, row, name, smem_optin)
        h = handle(rt, scenes, name)
        W, H, spp, depth = WORLDS[name][1]
        want, rays, want_acc = oracle_render(ob, scenes, name)
        where = f"{row} on {name}"
        # 1. pixel items, one pass
        got, st = _render(rt, h, W, H, spp, depth, group_cull=cull, sample_items=False)
        check_stats(where, st, v)
        assert st.launches == 1 and st.rays == rays, (where, st.launches, st.rays, rays)
        assert np.array_equal(got, want), f"{where}: {int((got != want).any(axis=2).sum())} pixels differ from the oracle"
        # 2. two fused passes into the float4 sums: the colour below the RGBA8 pack, bit for bit
        accum = torch.full((H, W, 4), 7.0, dtype=torch.float32, device="cuda")
        out = torch.zeros((H, W), dtype=torch.int32, device="cuda")
        torch.cuda.synchronize()
        st = rt.RenderStats()
        rt.render_device(h, rt.Options(spp, depth, passes=2, accum_out=True, group_cull=cull, sample_items=False),
                         W, H, out.data_ptr(), accum.data_ptr(), 0, st)
        check_stats(where + " (passes=2)", st, v)
        assert st.passes_fused == 2 and st.rays == rays, (where, st.passes_fused, st.rays, rays)
        acc = accum.cpu().numpy()
        bad = np.argwhere(_bits(acc) != _bits(want_acc))
        assert bad.size == 0, (f"{where}: {len(bad)} float4 sums differ from the oracle's, first at {bad[0].tolist()}: "
                               f"{acc[tuple(bad[0])]} vs {want_acc[tuple(bad[0])]}")
        assert np.array_equal(out.cpu().numpy().view(np.uint8).reshape(H, W, 4), want), where
        # 3. sample items
        got, st = _render(rt, h, W, H, spp, depth, group_cull=cull, sample_items=True)
        check_stats(where + " (sample items)", st, v)
        assert st.sample_items == 1 and st.rays == rays and np.array_equal(got, want), (where, st.rays, rays)


FAST_FRAME = (192, 108, 8)


def check_render_fast(rt, ob, scenes, row, smem_optin):
    """Bars of test_fast_math_kernel_is_statistically_equivalent against the exact kernel (which the exact rows prove
    equal to the oracle); the noise floor is two exact renders with seeds 1 and 2."""
    cull = MATRIX[row].cull
    for name in MATRIX[row].worlds:
        v = selected(ob, scenes, row, name, smem_optin)
        h = handle(rt, scenes, name)
        W, H, spp = FAST_FRAME
        depth = WORLDS[name][1][3]
        where = f"{row} on {name}"
        fast, st_f = _render(rt, h, W, H, spp, depth, seed=1, fast_math=True, group_cull=cull)
        check_stats(where, st_f, v)
        exact, st_e = _render(rt, h, W, H, spp, depth, seed=1, group_cull=cull)
        other, _ = _render(rt, h, W, H, spp, depth, seed=2, group_cull=cull)
        floor, r = _rmse(exact, other), _rmse(exact, fast)
        assert r <= 0.35 * floor, f"{where}: RMSE {r} against the exact kernel, noise floor {floor}"
        d = np.abs(exact.astype(int) - fast.astype(int)).max(axis=2)
        assert (d > 1).mean() <= 0.01, f"{where}: {(d > 1).mean():.4f} of the pixels differ by more than 1/255"
        assert abs(int(st_e.rays) - int(st_f.rays)) <= 1e-3 * st_e.rays, (where, st_e.rays, st_f.rays)
        if counts_of(ob, scenes, name).n_sph >= FILTER_FROM:           # the same filter test decides: bit-identical
            twin, st_t = _render(rt, h, W, H, spp, depth, seed=1, fast_math=True, group_cull=not cull)
            assert st_t.culled == int(not cull), where
            assert st_t.rays == st_f.rays and np.array_equal(twin, fast), f"{where}: fast CULL != fast FILTER"


def check_aov(rt, ob, scenes, row, smem_optin):
    cull = MATRIX[row].cull
    for name in MATRIX[row].worlds:
        v = selected(ob, scenes, row, name, smem_optin)
        cam, world = oracle_world(ob, scenes, name)
        W, H = 96, 54
        st = rt.RenderStats()
        got = rt.render_aov(handle(rt, scenes, name), W, H, rt.Options(group_cull=cull, sample_begin=1), st)
        check_stats(f"{row} on {name}", st, v)
        assert st.rays == W * H
        test_aov.assert_same({k: t.cpu().numpy() for k, t in got.items()},
                             test_aov.primary_hits(ob, world, cam, W, H, sample_begin=1), canonical_nan=True)


def _lane_rays(ob, scenes, row, name):
    cam, world = oracle_world(ob, scenes, name)
    return world, test_rays.families(ob, world, cam, seed=zlib.crc32(f"{row}/{name}".encode()) & 0xFFFF, n=64)


def check_ray(rt, ob, scenes, row, smem_optin):
    cull = MATRIX[row].cull
    for name in MATRIX[row].worlds:
        v = selected(ob, scenes, row, name, smem_optin)
        world, rays = _lane_rays(ob, scenes, row, name)
        st = rt.RenderStats()
        got = test_rays._gpu(rt, handle(rt, scenes, name), rays, cull, st)
        check_stats(f"{row} on {name}", st, v)
        assert st.rays == len(rays)
        test_rays.assert_same(got, test_rays.reference(ob, world, rays), canonical_nan=True)


def check_occlusion(rt, ob, scenes, row, smem_optin):
    cull = MATRIX[row].cull
    for name in MATRIX[row].worlds:
        v = selected(ob, scenes, row, name, smem_optin)
        world, rays = _lane_rays(ob, scenes, row, name)
        st = rt.RenderStats()
        got = test_occlusion._gpu(rt, handle(rt, scenes, name), rays, cull, st)
        check_stats(f"{row} on {name}", st, v)
        assert st.rays == len(rays)
        test_occlusion.assert_answers(got, test_occlusion.expected(ob, world, rays))


CHECKS = {"render-exact": check_render_exact, "render-fast": check_render_fast, "aov": check_aov, "ray": check_ray,
          "occlusion": check_occlusion}


def run_rows(rt, ob, scenes, rows) -> dict:
    """{row: None if it passed, else the failure's text}."""
    import traceback
    smem_optin, out = smem_optin_of_device(), {}
    for row in rows:
        try:
            CHECKS[key_of(row).kernel](rt, ob, scenes, row, smem_optin)
            out[row] = None
        except AssertionError:
            out[row] = traceback.format_exc(limit=3)
    return out


# ------------------------------------------------------------------------------------------------ switch points

def switch_worlds(smem_optin: int):
    """{case id: (S, T, cull, expected hot bytes, expected staged, expected block)}: for the DIRECT walk with triangles,
    FILTER and CULL, a world whose hot lists are exactly 57,344 bytes (the largest 256-thread staging), the next size up
    (1024 threads), exactly smem_optin - 1024 (the largest staging) and the next size up (global memory).  Every hot
    size is a multiple of 32 and a pair of triangles adds 32 bytes, so "next" is T + 2.  Synthetic worlds have one
    ground sphere above 8x the median radius: one "always" cull group."""
    limit = smem_optin - 1024
    assert limit % 32 == 0, f"smem_optin {smem_optin}: no world has hot lists of exactly {limit} bytes"
    out = {}
    for tag, target in (("57344", LARGE_SMEM_FROM), ("limit", limit)):
        # DIRECT: 16 (Sp + Tp) with 37 spheres (Sp = 40)
        Tp = target // 16 - 40
        out[f"DIRECT-tris-{tag}"] = (37, Tp - 1, False)
        # FILTER: 20 Sp + 16 Tp, Sp = 8a with most of the bytes in spheres
        Sp = 8 * int(0.95 * target // 160)
        Tp = (target - 20 * Sp) // 16
        out[f"FILTER-{tag}"] = (Sp - 3, Tp - 1, False)
        # CULL: 160 G + 16 Tp, G = 32g groups = 1 + ceil((S - 1) / 8)
        G = 32 * int(0.95 * target // 5120)
        Tp = (target - 160 * G) // 16
        out[f"CULL-{tag}"] = (8 * (G - 16) - 2, Tp - 1, True)
    cases_ = {}
    for cid, (S, T, cull) in out.items():
        walk, tag = cid.rsplit("-", 1)
        target = LARGE_SMEM_FROM if tag == "57344" else limit
        cases_[cid] = (S, T, cull, target, True, 256 if tag == "57344" else 1024)
        after = {"57344": ("57376", True, 1024), "limit": ("limit+32", False, 256)}[tag]
        cases_[f"{walk}-{after[0]}"] = (S, T + 2, cull, target + 32, after[1], after[2])
    return cases_


SWITCH_IDS = list(switch_worlds(B200_SMEM_OPTIN))


def _switch_world(ob, scenes, cid, smem_optin):
    S, T, cull, hot, staged, block = switch_worlds(smem_optin)[cid]
    name = f"switch-{S}-{T}"
    if name not in WORLDS:
        WORLDS[name] = (_syn(S, T, S + T), BIG)
    v = choose(counts_of(ob, scenes, name), cull, 1, smem_optin)
    assert (v.hot, v.smem, v.block) == (hot, staged, block), (cid, v)
    assert v.walk == WALKS[cid.split("-")[0]], (cid, v)
    return name, cull, v


# ===================================================================================================== CPU tests

def _kernels_in(obj: Path):
    """{mangled name} of the entry functions (kernels) of a built object."""
    out = subprocess.run(["cuobjdump", "-symbols", str(obj)], capture_output=True, text=True, check=True).stdout
    return {line.split()[-1] for line in out.splitlines() if "STO_ENTRY" in line}


MANGLED = re.compile(r"^_ZN2rt\d+rt_(render|aov|ray|occlusion)_kernelI((?:L[bi]\d+E)+)E")
NOT_WALKS = ("rt_resolve_samples_kernel", "rt_gather_rows_kernel", "rt_selftest_sqrt_kernel",
             "rt_selftest_division_kernel", "rt_ffma_peak_kernel")


def _demangle(name: str) -> str:
    if shutil.which("c++filt"):
        return subprocess.run(["c++filt", name], capture_output=True, text=True).stdout.strip() or name
    return name


def key_of_symbol(name: str):
    m = MANGLED.match(name)
    if not m:
        return None
    args = [int(a) for a in re.findall(r"L[bi](\d+)E", m[2])]
    if m[1] == "render":
        fast, smem, block, sph, tris, np_ = args
        return Key("render-fast" if fast else "render-exact", bool(smem), block, sph, bool(tris), np_)
    smem, block, sph, tris = args
    return Key(m[1], bool(smem), block, sph, bool(tris), 1)


@pytest.mark.skipif(shutil.which("cuobjdump") is None, reason="cuobjdump not installed")
def test_matrix_rows_are_exactly_the_built_instantiations():
    objs = [OBJ / "rt_kernels_exact.o", OBJ / "rt_kernels_fast.o"]
    if not all(o.exists() for o in objs):
        import __graft_entry__
        __graft_entry__.build()
    built, other = {}, []
    for o in objs:
        for name in _kernels_in(o):
            k = key_of_symbol(name)
            if k is not None:
                built[id_of(k)] = name
            elif not any(n in name for n in NOT_WALKS):
                other.append(_demangle(name))
    assert not other, f"kernels that are neither in the variant matrix nor known non-walk kernels: {other}"
    for row in MATRIX:
        assert id_of(key_of(row)) == row, f"row id {row!r} is not canonical"
    missing = sorted(set(built) - set(MATRIX))
    assert not missing, "instantiations without a row in MATRIX: " + "; ".join(
        f"{r} = {_demangle(built[r])}" for r in missing)
    stale = sorted(set(MATRIX) - set(built))
    assert not stale, f"rows of MATRIX that the objects do not instantiate: {stale}"
    assert len(built) == 102


def test_restatement_selects_every_run_row_on_b200(ob, scenes):
    for row in RUN_ROWS:
        assert MATRIX[row].worlds and all(w in WORLDS for w in MATRIX[row].worlds), row
        for name in MATRIX[row].worlds:
            selected(ob, scenes, row, name, B200_SMEM_OPTIN)
    # every reachable instantiation is run: 22 render rows of each policy, 16 of each lane kernel
    per = {k: sum(key_of(r).kernel == k for r in RUN_ROWS) for k in KERNELS}
    assert per == {"render-exact": 22, "render-fast": 22, "aov": 16, "ray": 16, "occlusion": 16}, per


def test_ragged_worlds_walk_the_pads(ob, scenes):
    """Apart from the 8-sphere scenes of the reference and the 64-sphere switch world, every sphere count is not a
    multiple of 8 and every triangle count is odd."""
    for name in WORLDS:
        if name.startswith("switch-"):
            continue
        c = counts_of(ob, scenes, name)
        _, world = oracle_world(ob, scenes, name)
        if name not in ("default", "example", "s64"):
            assert c.n_sph % 8 and c.n_sph_pad > c.n_sph, name
        if world.n_triangles and name != "example":
            assert c.n_tri_pad == world.n_triangles + 1, name


def test_unreachable_rows_are_unreachable():
    """A DIRECT world has at most 63 spheres; without triangles its hot lists are at most 64 x 16 bytes, whatever
    the cull flag, the paths per lane and the device, so it is always staged at 256 threads."""
    dead = {r for r, v in MATRIX.items() if isinstance(v, Unreachable)}
    want = {id_of(Key(k, smem, block, DIRECT, False, 1)) for k in KERNELS for smem, block in ((True, 1024), (False, 256))}
    assert dead == want and len(dead) == 10
    reached = set()
    for S in range(FILTER_FROM):
        for kernel in KERNELS:
            for cull in (False, True):
                for np_ in (1, 2):
                    for optin in (B200_SMEM_OPTIN, 48 * 1024 + 1024, 1024 + 1024):
                        c = packed_counts(np.full(S, 0.5, np.float32), 0)
                        v = choose(c, cull, np_, optin, lane_kernel=not kernel.startswith("render"))
                        assert v.hot <= 64 * 16 and v.walk == DIRECT
                        reached.add(id_of(key_for(kernel, v)))
    assert not (reached & dead)
    assert reached == {id_of(Key(k, True, 256, DIRECT, False, 1)) for k in KERNELS}


def test_restatement_of_the_pack():
    """The pad and cull-group rules on hand-made radii."""
    assert packed_counts([], 0) == Counts(0, 0, 0, 0)
    assert packed_counts(np.ones(63), 3) == Counts(63, 64, 4, 0)                  # no block C below 64 spheres
    assert packed_counts(np.ones(64), 0) == Counts(64, 64, 0, 32)
    r = np.ones(300, np.float32)
    r[:9] = 8.0                                                                   # 8x the median is not "large"
    assert packed_counts(r, 1).n_groups == 64                                     # ceil(300 / 8) = 38 -> 64
    r[:9] = 8.001
    assert packed_counts(r, 1) == Counts(300, 304, 2, 64)                         # 2 + 37 -> 64
    r = np.concatenate([np.full(270, 1000.0), np.ones(1000)])                    # 34 + 125 groups -> 160
    assert packed_counts(r, 0).n_groups == 160
    c = Counts(40, 40, 3544, 0)                                                   # 16 x 3584 = 57,344 bytes
    assert choose(c, False, 1, B200_SMEM_OPTIN) == Variant(True, 256, DIRECT, True, 57344, 1)
    assert choose(c._replace(n_tri_pad=3546), False, 2, B200_SMEM_OPTIN).block == 1024
    c = Counts(4001, 4008, 0, 512)
    assert choose(c, False, 2, B200_SMEM_OPTIN) == Variant(True, 512, FILTER, False, 80160, 2)
    assert choose(c, False, 2, B200_SMEM_OPTIN, lane_kernel=True).block == 1024
    assert choose(c, True, 2, B200_SMEM_OPTIN) == Variant(True, 1024, CULL, False, 81920, 1)


def test_switch_worlds_are_solved_for_b200(ob, scenes):
    assert len(SWITCH_IDS) == 12
    for cid in SWITCH_IDS:
        _switch_world(ob, scenes, cid, B200_SMEM_OPTIN)


# ===================================================================================================== GPU tests

@pytest.mark.gpu
@pytest.mark.parametrize("row", _rows(("render-exact",), False))
def test_render_exact(gpu_rt, ob, scenes, row):
    check_render_exact(gpu_rt, ob, scenes, row, smem_optin_of_device())


@pytest.mark.gpu
@pytest.mark.parametrize("row", _rows(("render-fast",), False))
def test_render_fast(gpu_rt, ob, scenes, row):
    check_render_fast(gpu_rt, ob, scenes, row, smem_optin_of_device())


@pytest.mark.gpu
@pytest.mark.parametrize("row", _rows(("aov",), False))
def test_first_hit(gpu_rt, ob, scenes, row):
    check_aov(gpu_rt, ob, scenes, row, smem_optin_of_device())


@pytest.mark.gpu
@pytest.mark.parametrize("row", _rows(("ray",), False))
def test_ray_query(gpu_rt, ob, scenes, row):
    check_ray(gpu_rt, ob, scenes, row, smem_optin_of_device())


@pytest.mark.gpu
@pytest.mark.parametrize("row", _rows(("occlusion",), False))
def test_occlusion_query(gpu_rt, ob, scenes, row):
    check_occlusion(gpu_rt, ob, scenes, row, smem_optin_of_device())


NP2_ROWS = _rows(("render-exact", "render-fast"), True)


@pytest.fixture(scope="module")
def two_path_results(gpu_rt, ob):
    """Every two-paths-per-lane row, checked in one process started with RT_PATHS_PER_LANE=2."""
    code = ("import json, sys\n"
            f"sys.path[:0] = [{str(ROOT)!r}, {str(ROOT / 'oracle')!r}, {str(ROOT / 'tests')!r}]\n"
            "import importlib, oracle_binding as ob, test_variant_matrix as m\n"
            "rt = importlib.import_module('rust-swift-raytracer_b200')\n"
            "scenes = importlib.import_module('rust-swift-raytracer_b200.scenes')\n"
            f"print('RESULTS ' + json.dumps(m.run_rows(rt, ob, scenes, {NP2_ROWS!r})))\n")
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=1800,
                       env=dict(os.environ, RT_PATHS_PER_LANE="2"), cwd=str(ROOT))
    lines = [l for l in r.stdout.splitlines() if l.startswith("RESULTS ")]
    assert r.returncode == 0 and lines, r.stdout[-4000:] + r.stderr[-4000:]
    return json.loads(lines[-1][len("RESULTS "):])


@pytest.mark.gpu
@pytest.mark.parametrize("row", NP2_ROWS)
def test_two_paths_per_lane(two_path_results, row):
    assert row in two_path_results, row
    assert two_path_results[row] is None, two_path_results[row]


@pytest.mark.gpu
@pytest.mark.parametrize("cid", SWITCH_IDS)
def test_switch_points(gpu_rt, ob, scenes, cid):
    """The worlds on choose_variant's switch points, solved for this device: the render's and the first-hit kernel's
    launch statistics, and both against their references."""
    rt, optin = gpu_rt, smem_optin_of_device()
    name, cull, v = _switch_world(ob, scenes, cid, optin)
    h = handle(rt, scenes, name)
    cam, world = oracle_world(ob, scenes, name)
    W, H, spp, depth = WORLDS[name][1]
    want, rays, _ = oracle_render(ob, scenes, name)
    got, st = _render(rt, h, W, H, spp, depth, group_cull=cull, sample_items=False)
    check_stats(cid, st, v)
    assert st.rays == rays and np.array_equal(got, want), cid
    st = rt.RenderStats()
    aov = rt.render_aov(h, 64, 36, rt.Options(group_cull=cull), st)
    check_stats(cid + " (first hit)", st, v)
    test_aov.assert_same({k: t.cpu().numpy() for k, t in aov.items()}, test_aov.primary_hits(ob, world, cam, 64, 36),
                         canonical_nan=True)
