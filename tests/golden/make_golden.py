"""Generate golden input/output vectors by running the UNMODIFIED reference (oracle/_ref/libembree4.so.4, built
from /root/reference by oracle/build_ref.py) in this container.  Committed outputs: tests/golden/*.npz.

    python tests/golden/make_golden.py

Each fixture holds the scene (vertices/indices per geometry, masks), the RTCRayHit inputs and the reference's
outputs for rtcIntersect1 and rtcOccluded1, plus rtcGetSceneBounds.  Scenes/rays are seeded and small so the
fixtures stay a few hundred KB.
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from embree_b200 import scenes  # noqa: E402
from embree_b200.rtc import RTCBounds, make_rayhits, rays_of  # noqa: E402
from tests.parity import load_reference  # noqa: E402
import ctypes as C  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))


def random_rays_box(n, lo, hi, seed):
    rng = np.random.RandomState(seed)
    org = rng.uniform(lo, hi, (n, 3)).astype(np.float32)
    d = rng.normal(size=(n, 3)).astype(np.float32)
    return org, d


def run(name, meshes, rayhits):
    d = run_flags(name, meshes, rayhits, 0)
    r = run_flags(name, meshes, rayhits, 4)   # RTC_SCENE_FLAG_ROBUST: Triangle4v + Pluecker (scene.cpp:181-188)
    d["intersect_out_robust"], d["occluded_out_robust"] = r["intersect_out"], r["occluded_out"]
    np.savez_compressed(os.path.join(HERE, name + ".npz"), **d)


def run_flags(name, meshes, rayhits, flags):
    R = load_reference()
    dev = R.new_device(None)
    sc = R.rtcNewScene(dev)
    if flags:
        R.rtcSetSceneFlags(sc, flags)
    keep = []
    for (v, t, gid, mask) in meshes:
        add = R.add_quad_mesh if t.shape[1] == 4 else R.add_triangle_mesh   # [n,4] indices: RTC_GEOMETRY_TYPE_QUAD
        _, k = add(dev, sc, v, t, mask=mask, geom_id=gid)
        keep.append(k)
    R.rtcCommitScene(sc)
    R.check(dev)
    b = RTCBounds()
    R.rtcGetSceneBounds(sc, C.byref(b))
    out_i = R.intersect(sc, rayhits.copy(), "1")
    occ = rays_of(rayhits)
    out_o = R.occluded(sc, occ, "1")
    out_16 = R.intersect(sc, rayhits.copy(), "16")
    assert (out_16["primID"] == out_i["primID"]).all(), "reference packet path disagrees with its single-ray path"
    R.check(dev)
    d = dict(rays_in=rayhits.view(np.uint8).reshape(-1, 96), intersect_out=out_i.view(np.uint8).reshape(-1, 96),
             occluded_out=out_o.view(np.uint8).reshape(-1, 48),
             bounds=np.array([b.lower_x, b.lower_y, b.lower_z, b.upper_x, b.upper_y, b.upper_z], np.float32),
             n_meshes=np.array(len(meshes)))
    for i, (v, t, gid, mask) in enumerate(meshes):
        d[f"v{i}"], d[f"t{i}"], d[f"gid{i}"], d[f"mask{i}"] = v, t, np.array(gid, np.uint32), np.array(mask, np.uint32)
    hits = (out_i["geomID"] != 0xFFFFFFFF).mean()
    print(f"{name} flags={flags}: {len(rayhits)} rays, hit rate {hits:.3f}, occluded {(out_o['tfar'] == -np.inf).mean():.3f}")
    R.rtcReleaseScene(sc)
    R.rtcReleaseDevice(dev)
    return d


def instance_transforms(n, seed):
    """n affine transforms (rotation * non-uniform scale + translation), 12 floats each: columns vx | vy | vz | p."""
    rng = np.random.RandomState(seed)
    out = []
    for _ in range(n):
        q, _r = np.linalg.qr(rng.normal(size=(3, 3)))
        m = (q * rng.uniform(0.5, 1.5, 3)).astype(np.float32)      # columns scaled
        p = rng.uniform(-4, 4, 3).astype(np.float32)
        out.append(np.concatenate([m.T.reshape(-1), p]).astype(np.float32))
    return np.stack(out)


def run_instances(name, child_meshes, top_meshes, xfms, inst_masks, rayhits):
    """Two-level scene (tutorials/instanced_geometry): `top_meshes` + one RTC_GEOMETRY_TYPE_INSTANCE of the child scene
    per row of xfms, attached after the meshes (geomIDs len(top_meshes)...)."""
    R = load_reference()
    dev = R.new_device(None)
    child = R.rtcNewScene(dev)
    keep = [R.add_triangle_mesh(dev, child, v, t, mask=mask, geom_id=gid)[1] for (v, t, gid, mask) in child_meshes]
    R.rtcCommitScene(child)
    top = R.rtcNewScene(dev)
    keep += [R.add_triangle_mesh(dev, top, v, t, mask=mask, geom_id=gid)[1] for (v, t, gid, mask) in top_meshes]
    first = max([g for (_, _, g, _) in top_meshes] + [-1]) + 1
    for i, m in enumerate(xfms):
        R.add_instance(dev, top, child, m, mask=int(inst_masks[i]), geom_id=first + i)
    R.rtcCommitScene(top)
    R.check(dev)
    b = RTCBounds()
    R.rtcGetSceneBounds(top, C.byref(b))
    out_i = R.intersect(top, rayhits.copy(), "1")
    out_o = R.occluded(top, rays_of(rayhits), "1")
    out_8 = R.intersect(top, rayhits.copy(), "8")
    assert (out_8["primID"] == out_i["primID"]).all() and (out_8["instID"] == out_i["instID"]).all()
    R.check(dev)
    d = dict(rays_in=rayhits.view(np.uint8).reshape(-1, 96), intersect_out=out_i.view(np.uint8).reshape(-1, 96),
             occluded_out=out_o.view(np.uint8).reshape(-1, 48),
             bounds=np.array([b.lower_x, b.lower_y, b.lower_z, b.upper_x, b.upper_y, b.upper_z], np.float32),
             n_child=np.array(len(child_meshes)), n_top=np.array(len(top_meshes)), xfms=xfms,
             inst_masks=np.asarray(inst_masks, np.uint32), first_inst=np.array(first, np.uint32))
    for pre, ms in (("c", child_meshes), ("m", top_meshes)):
        for i, (v, t, gid, mask) in enumerate(ms):
            d[f"{pre}v{i}"], d[f"{pre}t{i}"], d[f"{pre}gid{i}"], d[f"{pre}mask{i}"] = v, t, np.array(gid, np.uint32), np.array(mask, np.uint32)
    print(f"{name}: {len(rayhits)} rays, hit rate {(out_i['geomID'] != 0xFFFFFFFF).mean():.3f}, "
          f"instance hits {(out_i['instID'] != 0xFFFFFFFF).mean():.3f}, occluded {(out_o['tfar'] == -np.inf).mean():.3f}")
    np.savez_compressed(os.path.join(HERE, name + ".npz"), **d)
    R.rtcReleaseScene(top)
    R.rtcReleaseScene(child)
    R.rtcReleaseDevice(dev)


def run_curves(name, meshes, curves, rayhits):
    """Round linear curves (RTC_GEOMETRY_TYPE_ROUND_LINEAR_CURVE, tutorials/hair_geometry / curve_geometry) next to
    triangle meshes.  curves: list of (vertices[nv,4], first-vertex indices, flags or None, geomID, mask)."""
    R = load_reference()
    dev = R.new_device(None)
    sc = R.rtcNewScene(dev)
    keep = [R.add_triangle_mesh(dev, sc, v, t, mask=mask, geom_id=gid)[1] for (v, t, gid, mask) in meshes]
    keep += [R.add_round_linear_curves(dev, sc, c[0], c[1], c[2], mask=c[4], geom_id=c[3], flat=len(c) > 5 and c[5])[1] for c in curves]
    R.rtcCommitScene(sc)
    R.check(dev)
    b = RTCBounds()
    R.rtcGetSceneBounds(sc, C.byref(b))
    out_i = R.intersect(sc, rayhits.copy(), "1")
    out_o = R.occluded(sc, rays_of(rayhits), "1")
    out_8 = R.intersect(sc, rayhits.copy(), "8")
    assert (out_8["primID"] == out_i["primID"]).all() and (out_8["geomID"] == out_i["geomID"]).all()
    R.check(dev)
    d = dict(rays_in=rayhits.view(np.uint8).reshape(-1, 96), intersect_out=out_i.view(np.uint8).reshape(-1, 96),
             occluded_out=out_o.view(np.uint8).reshape(-1, 48),
             bounds=np.array([b.lower_x, b.lower_y, b.lower_z, b.upper_x, b.upper_y, b.upper_z], np.float32),
             n_meshes=np.array(len(meshes)), n_curves=np.array(len(curves)))
    for i, (v, t, gid, mask) in enumerate(meshes):
        d[f"v{i}"], d[f"t{i}"], d[f"gid{i}"], d[f"mask{i}"] = v, t, np.array(gid, np.uint32), np.array(mask, np.uint32)
    for i, c in enumerate(curves):
        cv, ci, cf, gid, mask = c[:5]
        d[f"cv{i}"], d[f"ci{i}"], d[f"cgid{i}"], d[f"cmask{i}"] = cv, ci, np.array(gid, np.uint32), np.array(mask, np.uint32)
        d[f"cf{i}"] = np.zeros(0, np.uint8) if cf is None else np.asarray(cf, np.uint8)
        d[f"cflat{i}"] = np.array(1 if (len(c) > 5 and c[5]) else 0)
    print(f"{name}: {len(rayhits)} rays, hit rate {(out_i['geomID'] != 0xFFFFFFFF).mean():.3f}, curve hits "
          f"{np.isin(out_i['geomID'], [c[3] for c in curves]).mean():.3f}, occluded {(out_o['tfar'] == -np.inf).mean():.3f}")
    np.savez_compressed(os.path.join(HERE, name + ".npz"), **d)
    R.rtcReleaseScene(sc)
    R.rtcReleaseDevice(dev)


def main_curves():
    # a fur ball around a triangle sphere (geomID 0), two curve sets: library-derived neighbour flags (geomID 1, masked) and
    # application flags that cut every strand into capped pieces (geomID 2)
    v, t = scenes.triangle_sphere(12)
    cv, ci, _ = scenes.hair_ball(160, 5, seed=3, width=0.03)
    cv2, ci2, _ = scenes.hair_ball(40, 4, seed=8, radius=1.0, length=0.6, width=0.06)
    fl2 = np.tile(np.array([0, 2, 1, 0], np.uint8), 40)          # per strand: lone segment, a pair, lone segment
    rng = np.random.RandomState(11)
    org = rng.normal(size=(6000, 3)).astype(np.float32)
    org = org / np.linalg.norm(org, axis=1, keepdims=True) * rng.uniform(1.05, 2.5, (6000, 1)).astype(np.float32)
    d = (-org + rng.normal(scale=0.6, size=org.shape)).astype(np.float32)
    rays = make_rayhits(org, d)
    rays["tnear"][::7] = 0.3
    rays["tfar"][::5] = 1.2
    rays["mask"][::3] = 0x2
    rays["id"] = np.arange(len(rays))
    run_curves("curves", [(v, t, 0, 0xFFFFFFFF)], [(cv, ci, None, 1, 0x3), (cv2, ci2, fl2, 2, 0xFFFFFFFD)], rays)
    # the same kind of scene with RTC_GEOMETRY_TYPE_FLAT_LINEAR_CURVE sets (ray-facing ribbons), un-normalised ray directions
    cv3, ci3, _ = scenes.hair_ball(200, 5, seed=13, width=0.03)
    rays2 = rays.copy()
    scale = rng.uniform(0.3, 4.0, len(rays2)).astype(np.float32)
    for f in ("dir_x", "dir_y", "dir_z"):
        rays2[f] *= scale
    rays2["tnear"] = 0.0
    rays2["tfar"] = np.inf
    rays2["tfar"][::5] = 1.2 / scale[::5]
    run_curves("curves_flat", [(v, t, 0, 0xFFFFFFFF)], [(cv3, ci3, None, 1, 0x3, True), (cv2, ci2, None, 2, 0xFFFFFFFD, True)], rays2)


from tests.golden.make_golden_sets import CUBIC_SETS  # noqa: E402


def main_cubic_curves(name="curves_cubic", rnd=False):
    """Flat cubic curves (curve_intersector_ribbon.h; rnd: ROUND cubic curves, curve_intersector_sweep.h): one curve set per basis,
    each with its own tessellation rate and geometry mask, around a triangle sphere; rays from outside towards the ball, some
    with masks and tnear / tfar windows."""
    R = load_reference()
    v, t = scenes.triangle_sphere(12)
    v = (v * np.float32(0.9)).astype(np.float32)
    sets = []
    for k, (basis, tess) in enumerate(CUBIC_SETS):
        cv, ci, tg = scenes.cubic_hair(60, basis, seed=20 + k, radius=0.9, width=0.03)
        sets.append((cv, ci, 1 + k, 0xFFFFFFFF if k != 2 else 0x6, basis, tess, tg))
    rng = np.random.RandomState(31)
    org = rng.normal(size=(6144, 3)).astype(np.float32)
    org = org / np.linalg.norm(org, axis=1, keepdims=True) * rng.uniform(1.5, 2.5, (6144, 1)).astype(np.float32)
    d = (-org + rng.normal(scale=0.45, size=org.shape)).astype(np.float32)
    rays = make_rayhits(org, d)
    rays["mask"][0::7] = 0x2
    rays["mask"][1::7] = 0x1
    rays["tnear"][2::9] = 1.2
    rays["tfar"][3::11] = 1.6
    rays["id"] = np.arange(len(rays))
    dev = R.new_device(None)
    sc = R.rtcNewScene(dev)
    keep = [R.add_triangle_mesh(dev, sc, v, t, mask=0xFFFFFFFF, geom_id=0)[1]]
    for (cv, ci, gid, mask, basis, tess, tg) in sets:
        keep.append(R.add_flat_cubic_curves(dev, sc, cv, ci, basis, tess, tg, mask=mask, geom_id=gid, round=rnd)[1])
    R.rtcCommitScene(sc)
    R.check(dev)
    b = RTCBounds()
    R.rtcGetSceneBounds(sc, C.byref(b))
    out_i = R.intersect(sc, rays.copy(), "1")
    out_o = R.occluded(sc, rays_of(rays), "1")
    R.check(dev)
    dd = dict(rays_in=rays.view(np.uint8).reshape(-1, 96), intersect_out=out_i.view(np.uint8).reshape(-1, 96),
              occluded_out=out_o.view(np.uint8).reshape(-1, 48),
              bounds=np.array([b.lower_x, b.lower_y, b.lower_z, b.upper_x, b.upper_y, b.upper_z], np.float32),
              v0=v, t0=t, n_sets=np.array(len(sets)), round=np.array(1 if rnd else 0))
    for i, (cv, ci, gid, mask, basis, tess, tg) in enumerate(sets):
        dd[f"cv{i}"], dd[f"ci{i}"], dd[f"cgid{i}"], dd[f"cmask{i}"] = cv, ci, np.array(gid, np.uint32), np.array(mask, np.uint32)
        dd[f"ctess{i}"] = np.array(0 if tess is None else tess)
        dd[f"ctang{i}"] = tg if tg is not None else np.zeros((0, 4), np.float32)
    np.savez_compressed(os.path.join(HERE, name + ".npz"), **dd)
    per = {basis: int((out_i["geomID"] == 1 + k).sum()) for k, (basis, _t) in enumerate(CUBIC_SETS)}
    print(f"{name}: {len(rays)} rays, hits per basis {per}, triangles {(out_i['geomID'] == 0).sum()}, occluded {(out_o['tfar'] == -np.inf).mean():.3f}")
    R.rtcReleaseScene(sc)
    R.rtcReleaseDevice(dev)


def main_filters():
    """Filter callbacks (tests/filter_cases.py) on the cube_ground scene: the reference's results with a geometry filter,
    the arguments' filter on every geometry, and the arguments' filter enabled on one geometry."""
    from tests import filter_cases as fc
    from tests.conftest import load_golden
    meshes, rin, _wi, _wo, _b = load_golden("cube_ground")
    R = load_reference()
    dev = R.new_device(None)
    d = {}
    for cfg in fc.CONFIGS:
        oi, oo, ri, ro = fc.run_config(R, dev, meshes, rin, cfg, "1")
        o16, oo16, r16, _q = fc.run_config(R, dev, meshes, rin, cfg, "16")
        if cfg == "argument_all":
            # Reference quirk: its PACKET intersectors are picked at commit (accel.h:240-253, scene.cpp:801
            # accels_select(hasFilterFunction())); when no geometry carries or enables a filter the "nofilter" variants
            # run and RTC_RAY_QUERY_FLAG_INVOKE_ARGUMENT_FILTER is ignored by rtcIntersect4/8/16.  The single-ray entry
            # point honours the flag as documented (context.h:48-50, filter.h:25-28): that is the golden behaviour.
            assert len(r16.calls) == 0
        else:
            assert (o16["primID"] == oi["primID"]).all() and (oo16["tfar"].view(np.uint32) == oo["tfar"].view(np.uint32)).all()
        d[cfg + "_intersect"], d[cfg + "_occluded"] = oi.view(np.uint8).reshape(-1, 96), oo.view(np.uint8).reshape(-1, 48)
        rej = sum(1 for c in ri.calls if fc.rejects(c[1], c[2], c[3]))
        print(f"filters/{cfg}: {len(ri.calls)} intersect callbacks ({rej} rejected), {len(ro.calls)} occluded callbacks, "
              f"hit rate {(oi['geomID'] != 0xFFFFFFFF).mean():.3f}, occluded {(oo['tfar'] == -np.inf).mean():.3f}")
    T, occ = fc.run_hair_shadows(R, dev)
    d["hair_T"], d["hair_occluded"] = T, occ
    print(f"filters/hair shadows: {len(occ)} rays, occluded {occ.mean():.3f}, partially transparent {((T < 1).any(1) & ~occ).mean():.3f}")
    R.rtcReleaseDevice(dev)
    np.savez_compressed(os.path.join(HERE, "filters.npz"), **d)


from tests.golden.make_golden_sets import point_scene  # noqa: E402


def main_points(name="points"):
    """Point primitives (RTC_GEOMETRY_TYPE_SPHERE_POINT / _DISC_POINT / _ORIENTED_DISC_POINT: sphere_intersector.h, disc_intersector.h)."""
    R = load_reference()
    dev = R.new_device(None)
    meshes, sets, rayhits = point_scene()
    sc = R.rtcNewScene(dev)
    keep = [R.add_triangle_mesh(dev, sc, v, t, mask=mask, geom_id=gid)[1] for (v, t, gid, mask) in meshes]
    keep += [R.add_points(dev, sc, pv, kind, normals=pn, mask=mask, geom_id=gid)[1] for (pv, kind, pn, gid, mask) in sets]
    R.rtcCommitScene(sc)
    R.check(dev)
    b = RTCBounds()
    R.rtcGetSceneBounds(sc, C.byref(b))
    out_i = R.intersect(sc, rayhits.copy(), "1")
    out_o = R.occluded(sc, rays_of(rayhits), "1")
    out_8 = R.intersect(sc, rayhits.copy(), "8")
    assert (out_8["primID"] == out_i["primID"]).all() and (out_8["geomID"] == out_i["geomID"]).all()
    R.check(dev)
    d = dict(rays_in=rayhits.view(np.uint8).reshape(-1, 96), intersect_out=out_i.view(np.uint8).reshape(-1, 96),
             occluded_out=out_o.view(np.uint8).reshape(-1, 48),
             bounds=np.array([b.lower_x, b.lower_y, b.lower_z, b.upper_x, b.upper_y, b.upper_z], np.float32))
    print(f"{name}: {len(rayhits)} rays, hits per geometry {[int((out_i['geomID'] == g).sum()) for g in range(4)]}, "
          f"occluded {(out_o['tfar'] == -np.inf).mean():.3f}")
    np.savez_compressed(os.path.join(HERE, name + ".npz"), **d)
    R.rtcReleaseScene(sc)
    R.rtcReleaseDevice(dev)


def main():
    # 1. the triangle_geometry tutorial scene: cube (geomID 0) + ground plane (geomID 1), camera-like + random rays
    (cv, ct), (gv, gt) = scenes.cube_and_ground()
    prim = scenes.as_numpy_rayhits(scenes.primary_rays(48, 32, eye=(1.5, 1.5, -1.5), look=(-1.5, -1.5, 1.5), fov=90.0))
    org, d = random_rays_box(1024, -3, 3, 1)
    rnd = make_rayhits(org, d)
    both = np.concatenate([prim, rnd]).view(prim.dtype)
    both["id"] = np.arange(len(both))
    run("cube_ground", [(cv, ct, 0, 0xFFFFFFFF), (gv, gt, 1, 0xFFFFFFFF)], both)
    # 2. small sphere seen from inside (reference "incoherent" definition) and from outside, with tnear/tfar windows
    v, t = scenes.triangle_sphere(21)
    a = scenes.as_numpy_rayhits(scenes.incoherent_rays_reference(1536))
    org, d = random_rays_box(1024, -2, 2, 2)
    b = make_rayhits(org, d)
    b["tnear"][::3] = 0.5
    b["tfar"][::5] = 1.5
    ab = np.concatenate([a, b]).view(a.dtype)
    run("sphere21", [(v, t, 0, 0xFFFFFFFF)], ab)
    # 3. terrain with grazing rays + a second, masked geometry (ray masks select which one is visible)
    tv, tt = scenes.terrain(24, seed=3)
    pv, pt = scenes.triangle_plane((-1, 0.05, -1), (2, 0, 0), (0, 0, 2), 3, 3)
    org, d = random_rays_box(2048, -1, 1, 4)
    org[:, 1] = np.abs(org[:, 1]) * 0.3 + 0.2
    d[:, 1] = -np.abs(d[:, 1]) * 0.3
    r = make_rayhits(org, d)
    r["mask"][0::4] = 0x1
    r["mask"][1::4] = 0x2
    r["mask"][2::4] = 0x4
    r["mask"][3::4] = 0x3
    run("terrain_masks", [(tv, tt, 0, 0x1), (pv, pt, 3, 0x2)], r)
    # 3b. quad meshes (non-planar height-field quads, a closed quad box with one triangle-as-quad) next to a triangle
    #     mesh, with geometry masks; rays from above, from inside the box and at random
    qv, qq = scenes.quad_terrain(20, seed=5)
    bv = np.array([[x, y, z] for x in (-0.5, 0.5) for y in (0.3, 0.9) for z in (-0.5, 0.5)], np.float32)
    bq = np.array([[0, 1, 3, 2], [4, 6, 7, 5], [0, 4, 5, 1], [2, 3, 7, 6], [0, 2, 6, 4], [1, 5, 7, 7]], np.uint32)  # last: triangle as quad
    sv, st = scenes.triangle_sphere(8)
    sv = (sv * np.float32(0.25) + np.float32([0.0, 0.6, 0.0])).astype(np.float32)
    org, d = random_rays_box(3072, -1, 1, 6)
    org[:1024, 1] = 1.5
    d[:1024, 1] = -np.abs(d[:1024, 1]) - 0.2
    org[1024:2048] = org[1024:2048] * np.float32(0.2) + np.float32([0, 0.6, 0])
    r = make_rayhits(org, d)
    r["mask"][0::6] = 0x1
    r["mask"][1::6] = 0x2
    r["id"] = np.arange(len(r))
    run("quads", [(qv, qq, 0, 0x1), (bv, bq, 1, 0xFFFFFFFF), (sv, st, 2, 0x3)], r)
    # 4. single-level instancing: a ground plane + 7 transformed instances of a two-mesh child scene, with instance and
    #    geometry masks selecting subsets
    sv, st = scenes.triangle_sphere(10)
    sv2 = (sv * np.float32(0.5) + np.float32([1.2, 0, 0])).astype(np.float32)
    gv, gt = scenes.triangle_plane((-8, -3, -8), (16, 0, 0), (0, 0, 16), 4, 4)
    xf = instance_transforms(7, 11)
    org, d = random_rays_box(4096, -6, 6, 12)
    r = make_rayhits(org, d)
    r["mask"][0::5] = 0x2
    r["mask"][1::5] = 0x4
    r["tnear"][2::7] = 1.0
    r["id"] = np.arange(len(r))
    run_instances("instances", [(sv, st, 0, 0xFFFFFFFF), (sv2, st, 1, 0x3)], [(gv, gt, 0, 0xFFFFFFFF)], xf,
                  [0xFFFFFFFF if i % 3 else 0x5 for i in range(7)], r)
    main_curves()
    main_cubic_curves()
    main_cubic_curves("curves_cubic_round", True)
    main_points()
    main_filters()


def main_abi():
    """reference_abi.json: tests/test_abi.py's layout probe compiled against the reference headers (with the rtcore_config.h that
    oracle/build_ref.py generates) and the prototypes of every rtc* function they declare; the reference is where
    oracle/build_ref.py finds it."""
    import glob
    import json
    from tests import test_abi
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    from build_ref import REF as ref_dir
    probe = test_abi._probe("embree4/rtcore.h", extra_inc=(os.path.join(ref_dir, "include"),
                                                          os.path.join(ROOT, "oracle", "_ref", "gen_rel", "include", "embree4")))
    protos = {}
    for f in sorted(glob.glob(os.path.join(ref_dir, "include", "embree4", "*.h"))):
        protos.update(test_abi._prototypes(open(f).read()))
    rows = [f"  {json.dumps(k)}: {json.dumps(list(v))}" for k, v in sorted(protos.items())]
    with open(os.path.join(HERE, "reference_abi.json"), "w") as f:
        f.write('{"layout_probe": ' + json.dumps(probe) + ',\n "prototypes": {\n' + ",\n".join(rows) + "\n }}\n")


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "abi":
        main_abi()
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "curves":
        main_curves()
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "cubic":
        main_cubic_curves()
        main_cubic_curves("curves_cubic_round", True)
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "points":
        main_points()
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "filters":
        main_filters()
        sys.exit(0)
    if load_reference() is None:
        sys.exit("oracle/_ref/libembree4.so.4 missing: run python oracle/build_ref.py first")
    torch.manual_seed(0)
    main()
