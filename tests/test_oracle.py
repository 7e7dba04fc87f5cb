"""The oracle (oracle/embree_oracle.c, a scalar restatement of the reference hot path) is pinned here against
(1) the reference's own known-answer tests restated from tutorials/verify/verify.cpp, (2) golden vectors produced
by the unmodified reference (tests/golden/*.npz, tests/golden/make_golden.py) and (3) the reference library itself
when oracle/_ref has been built in this container."""
import numpy as np
import pytest

from embree_b200 import scenes
from embree_b200.rtc import make_rayhits, rays_of
from tests.conftest import GOLDEN, GOLDEN_QUADS, load_golden, load_golden_instances
from tests.parity import compare_hits, reference_run, sample_rays


def test_triangle_hit_kat(oracle):
    """TriangleHitTest (verify.cpp:2462-2547): 256 rays from z=-1 onto the unit triangle; geomID=0, primID=0,
    u,v,t within 16 ulp, Ng == (0,0,1), org+t*dir == v0+u(v1-v0)+v(v2-v0)."""
    v = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0]], np.float32)
    t = np.array([[0, 1, 2]], np.uint32)
    u0, v0 = np.meshgrid((np.arange(16) + 0.5) / 16 * 0.45, (np.arange(16) + 0.5) / 16 * 0.45)  # stays inside, off the edges
    org = np.stack([u0.ravel(), v0.ravel(), -np.ones(256)], 1).astype(np.float32)
    r = make_rayhits(org, np.tile([[0, 0, 1]], (256, 1)))
    out = oracle.trace(v, t, r)
    ulp = 16 * np.finfo(np.float32).eps
    assert (out["geomID"] == 0).all() and (out["primID"] == 0).all()
    assert np.abs(out["u"] - org[:, 0]).max() <= ulp and np.abs(out["v"] - org[:, 1]).max() <= ulp
    assert np.abs(out["tfar"] - 1.0).max() <= ulp
    assert (out["Ng_x"] == 0).all() and (out["Ng_y"] == 0).all() and (out["Ng_z"] == 1).all()
    assert (out["instID"] == 0xFFFFFFFF).all()


def test_minimal_tutorial_kat(oracle):
    """tutorials/minimal/minimal.cpp:159-206: ray (0.33,0.33,-1)+(0,0,1) hits at t=1; ray from (1,1,-1) misses."""
    v = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0]], np.float32)
    t = np.array([[0, 1, 2]], np.uint32)
    out = oracle.trace(v, t, make_rayhits([[0.33, 0.33, -1], [1, 1, -1]], [[0, 0, 1], [0, 0, 1]]))
    assert out["geomID"][0] == 0 and out["primID"][0] == 0 and out["tfar"][0] == 1.0
    assert abs(out["u"][0] - 0.33) < 1e-6 and abs(out["v"][0] - 0.33) < 1e-6
    assert out["geomID"][1] == 0xFFFFFFFF and np.isinf(out["tfar"][1])


@pytest.mark.parametrize("robust", [False, True])
@pytest.mark.parametrize("name", GOLDEN + GOLDEN_QUADS)
def test_oracle_vs_golden(oracle, name, robust):
    meshes, rin, want_i, want_o, bounds = load_golden(name, robust)
    sc = oracle.scene(meshes, robust=robust)
    got = sc.trace(rin.copy())
    rep = compare_hits(want_i, got)
    assert rep["id_mismatch"] == 0 and rep["tie"] == 0 and rep["hit_miss_disagree"] == 0, rep
    assert rep["max_rel_t"] <= 1e-4 and rep["max_abs_uv"] <= 1e-4 and rep["ng_bit_exact"] and rep["miss_untouched"], rep
    occ = sc.trace(rays_of(rin), occluded=True)
    assert (occ["tfar"].view(np.uint32) == want_o["tfar"].view(np.uint32)).all()
    assert np.array_equal(sc.bounds(), bounds)
    sc.free()


def oracle_instanced_scene(oracle, g):
    child = oracle.scene(g["child"])
    top = oracle.scene(g["top"], instances=[(child, m, g["first_inst"] + i, int(g["inst_masks"][i])) for i, m in enumerate(g["xfms"])])
    return top, child


def test_oracle_instances_vs_golden(oracle):
    """Single-level instancing (instance_intersector.cpp:15-67) against the reference's outputs: ids (incl. instID) and
    the object-space Ng exact; t/u/v agree to an ulp or two."""
    g = load_golden_instances()
    top, child = oracle_instanced_scene(oracle, g)
    got = top.trace(g["rays_in"].copy())
    want = g["intersect_out"]
    rep = compare_hits(want, got)
    assert (want["instID"] != 0xFFFFFFFF).sum() > 200
    assert rep["id_mismatch"] == 0 and rep["tie"] == 0 and rep["hit_miss_disagree"] == 0, rep
    assert rep["max_rel_t"] <= 1e-6 and rep["max_abs_uv"] <= 1e-6 and rep["ng_bit_exact"] and rep["miss_untouched"], rep
    assert (got["instPrimID"] == want["instPrimID"]).all()
    occ = top.trace(rays_of(g["rays_in"]), occluded=True)
    assert (occ["tfar"].view(np.uint32) == g["occluded_out"]["tfar"].view(np.uint32)).all()
    assert np.array_equal(top.bounds(), g["bounds"])
    top.free()
    child.free()


def test_oracle_vs_reference_live(oracle):
    v, t = scenes.triangle_sphere(41)
    rays = sample_rays(scenes.as_numpy_rayhits(scenes.incoherent_rays_reference(20000)))

    def run(R):
        dev = R.new_device(None)
        sc = R.rtcNewScene(dev)
        _, keep = R.add_triangle_mesh(dev, sc, v, t, mask=0xFFFFFFFF)
        R.rtcCommitScene(sc)
        out = R.intersect(sc, rays.copy(), "1"), R.occluded(sc, rays_of(rays), "1"), {}
        R.rtcReleaseScene(sc)
        R.rtcReleaseDevice(dev)
        return out
    want, wocc, _ = reference_run("triangle_sphere", rays, run)
    got = oracle.trace(v, t, rays.copy())
    rep = compare_hits(want, got)
    assert rep["id_mismatch"] == 0 and rep["hit_miss_disagree"] == 0 and rep["max_rel_t"] <= 1e-4 and rep["ng_bit_exact"], rep


def test_invalid_triangles_are_dropped(oracle):
    """scene_triangle_mesh.h:194-215: out-of-range index or non-finite / huge vertex drops the triangle."""
    v = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0], [np.nan, 0, 0], [2e18, 0, 0]], np.float32)
    t = np.array([[0, 1, 2], [0, 1, 3], [0, 1, 4], [0, 1, 7]], np.uint32)
    sc = oracle.scene([(v, t, 0, 0xFFFFFFFF)])
    assert sc.stats()["prims"] == 1
    out = sc.trace(make_rayhits([[0.2, 0.2, -1]], [[0, 0, 1]]))
    assert out["primID"][0] == 0
    sc.free()


def test_empty_scene(oracle):
    sc = oracle.scene([(np.zeros((0, 3), np.float32), np.zeros((0, 3), np.uint32), 0, 1)])
    out = sc.trace(make_rayhits([[0, 0, -1]], [[0, 0, 1]]))
    assert out["geomID"][0] == 0xFFFFFFFF and np.isinf(out["tfar"][0])
    sc.free()


@pytest.mark.parametrize("robust", [False, True])
def test_oracle_quads_and_instances_vs_reference_live(oracle, robust):
    """Randomised scenes beyond the golden fixtures, side by side with the reference's outputs: a
    quad mesh (non-planar quads, a triangle-as-quad, an invalid quad), a triangle mesh and four instances of a child
    scene that itself mixes quads and triangles, with geometry / instance / ray masks."""
    rng = np.random.RandomState(11 + robust)
    qv, qq = scenes.quad_terrain(24, seed=4)
    qq = qq.copy()
    qq[3, 3] = qq[3, 2]                      # triangle as quad
    qq[7] = (0, 1, 2, 0x7FFFFFF0)            # invalid index: dropped whole
    sv, st = scenes.triangle_sphere(9)
    sv = (sv * np.float32(0.3) + np.float32([0.2, 0.5, -0.1])).astype(np.float32)
    cv, cq = scenes.quad_terrain(6, seed=8)
    cv = (cv * np.float32(0.4)).astype(np.float32)
    xf = []
    for i in range(4):
        q, _ = np.linalg.qr(rng.normal(size=(3, 3)))
        m = (q * rng.uniform(0.5, 1.5, 3)).astype(np.float32)
        xf.append(np.concatenate([m.T.reshape(-1), rng.uniform(-1, 1, 3) + (0, 0.8, 0)]).astype(np.float32))
    imask = [0xFFFFFFFF, 0x1, 0x6, 0xFFFFFFFF]
    flags = 4 if robust else 0
    org = rng.uniform(-1.2, 1.2, (30000, 3)).astype(np.float32)
    org[:, 1] = np.abs(org[:, 1]) + 0.3
    rays = make_rayhits(org, rng.normal(size=(30000, 3)).astype(np.float32))
    rays["mask"][0::4] = 0x1
    rays["mask"][1::4] = 0x2
    rays["mask"][2::4] = 0x4
    rays = sample_rays(rays)

    def run(R):
        dev = R.new_device(None)
        child = R.rtcNewScene(dev)
        if flags:
            R.rtcSetSceneFlags(child, flags)
        keep = [R.add_quad_mesh(dev, child, cv, cq, mask=0x3, geom_id=0)[1], R.add_triangle_mesh(dev, child, sv * np.float32(0.5), st, mask=0xFFFFFFFF, geom_id=1)[1]]
        R.rtcCommitScene(child)
        top = R.rtcNewScene(dev)
        if flags:
            R.rtcSetSceneFlags(top, flags)
        keep += [R.add_quad_mesh(dev, top, qv, qq, mask=0x5, geom_id=0)[1], R.add_triangle_mesh(dev, top, sv, st, mask=0xFFFFFFFF, geom_id=1)[1]]
        for i, m in enumerate(xf):
            R.add_instance(dev, top, child, m, mask=imask[i], geom_id=2 + i)
        R.rtcCommitScene(top)
        R.check(dev)
        out = R.intersect(top, rays.copy(), "1"), R.occluded(top, rays_of(rays), "1"), {}
        R.rtcReleaseScene(top)
        R.rtcReleaseScene(child)
        R.rtcReleaseDevice(dev)
        del keep
        return out
    want, wocc, _ = reference_run(f"quads_instances{'_robust' if robust else ''}", rays, run)
    assert all((rays["mask"] == m).sum() > len(rays) // 8 for m in (0x1, 0x2, 0x4, 0xFFFFFFFF))   # every ray-mask class is traced
    oc = oracle.scene([(cv, cq, 0, 0x3), (sv * np.float32(0.5), st, 1, 0xFFFFFFFF)], robust=robust)
    ot = oracle.scene([(qv, qq, 0, 0x5), (sv, st, 1, 0xFFFFFFFF)], robust=robust,
                      instances=[(oc, m, 2 + i, imask[i]) for i, m in enumerate(xf)])
    got = ot.trace(rays.copy())
    rep = compare_hits(want, got, 1e-5)
    assert rep["hits"] > len(rays) // 10 and (want["instID"] != 0xFFFFFFFF).sum() > len(rays) // 100
    assert rep["id_mismatch"] == 0 and rep["hit_miss_disagree"] == 0 and rep["tie"] <= 2, rep
    assert rep["max_rel_t"] <= 1e-5 and rep["max_abs_uv"] <= 1e-5, rep
    gocc = ot.trace(rays_of(rays), occluded=True)
    assert (gocc["tfar"].view(np.uint32) == wocc["tfar"].view(np.uint32)).all()
    ot.free()
    oc.free()


@pytest.mark.parametrize("name", ["curves", "curves_flat"])
def test_oracle_curves_vs_golden(oracle, name):
    """Round linear curves (roundline_intersector.h) and flat linear curves (line_intersector.h) restated in
    oracle/embree_oracle.c against the reference's own outputs: two curve sets (library-derived and application neighbour
    flags, geometry masks) around a triangle sphere."""
    from tests.conftest import load_golden_curves
    g = load_golden_curves(name)
    sc = oracle.scene(g["meshes"], curves=g["curves"])
    got = sc.trace(g["rays_in"].copy())
    rep = compare_hits(g["intersect_out"], got)
    assert rep["id_mismatch"] == 0 and rep["hit_miss_disagree"] == 0 and rep["tie"] <= 40, rep    # ties: the joint of two segments
    assert rep["max_rel_t"] <= 1e-4 and rep["max_abs_uv"] <= 1e-4 and rep["miss_untouched"], rep
    ok = (got["geomID"] == g["intersect_out"]["geomID"]) & (got["primID"] == g["intersect_out"]["primID"]) & (got["geomID"] != 0xFFFFFFFF)
    for f in ("Ng_x", "Ng_y", "Ng_z"):
        assert np.allclose(got[f][ok], g["intersect_out"][f][ok], rtol=1e-3, atol=1e-5), f
    occ = sc.trace(rays_of(g["rays_in"]), occluded=True)
    assert (occ["tfar"].view(np.uint32) == g["occluded_out"]["tfar"].view(np.uint32)).all()
    assert np.array_equal(sc.bounds(), g["bounds"])
    sc.free()


def test_oracle_curves_vs_reference_live(oracle):
    """Larger randomised check against the reference's outputs: 3000 segments with neighbours, thin and thick."""
    from tests.parity import api_trace_mt
    cv, ci, cf = scenes.hair_ball(500, 6, seed=5, width=0.015)
    v, t = scenes.triangle_sphere(16)
    rng = np.random.RandomState(2)
    org = rng.normal(size=(60000, 3)).astype(np.float32)
    org = org / np.linalg.norm(org, axis=1, keepdims=True) * 2.5
    d = (-org + rng.normal(scale=0.5, size=org.shape)).astype(np.float32)
    rays = sample_rays(make_rayhits(org, d))
    sc = oracle.scene([(v, t, 0, 0xFFFFFFFF)], curves=[(cv, ci, cf, 1, 0xFFFFFFFF)])
    want = sc.trace(rays.copy(), nthreads=4)

    def run(R):
        dev = R.new_device(None)
        rs = R.rtcNewScene(dev)
        keep = [R.add_triangle_mesh(dev, rs, v, t, mask=0xFFFFFFFF, geom_id=0)[1], R.add_round_linear_curves(dev, rs, cv, ci, cf, mask=0xFFFFFFFF, geom_id=1)[1]]
        R.rtcCommitScene(rs)
        R.check(dev)
        out = api_trace_mt(R, rs, rays.copy(), 4), api_trace_mt(R, rs, rays_of(rays), 4, occluded=True), {}
        R.rtcReleaseScene(rs)
        R.rtcReleaseDevice(dev)
        del keep
        return out
    ref, ro, _ = reference_run("curves_round_linear", rays, run)
    from tests.parity import unexplained_curve_disagreements
    rep = compare_hits(ref, want)
    n_differ, unexplained = unexplained_curve_disagreements(rays, ref, want, {1: (cv, ci)})
    # a ray tangent to a cone flips between hit and miss with the rounding of the discriminant: every disagreement must be one
    assert (ref["geomID"] == 1).sum() > len(rays) // 20 and n_differ <= 6 and unexplained == 0, (rep, n_differ, unexplained)
    assert rep["max_rel_t"] <= 1e-4 and rep["max_abs_uv"] <= 2e-4, rep
    wo = sc.trace(rays_of(rays), occluded=True, nthreads=4)
    assert ((ro["tfar"] < 0) != (wo["tfar"] < 0)).sum() <= n_differ
    sc.free()


@pytest.mark.parametrize("name", ["curves_cubic", "curves_cubic_round"])
def test_oracle_cubic_curves_vs_golden(oracle, name):
    """Flat Bezier / B-spline / Catmull-Rom / Hermite curves (curve_intersector_ribbon.h:73-190, tessellation rates 4 / 7 / 4 / 12)
    and their ROUND counterparts (curve_intersector_sweep.h) restated in oracle/embree_oracle.c against the reference's own
    outputs: ids exact, t / u / v and Ng within tolerance, any-hit equal, scene bounds equal."""
    from tests.conftest import load_golden_cubic
    g = load_golden_cubic(name)
    rnd = name.endswith("round")
    sc = oracle.scene(g["meshes"], cubics=[(c[0], c[1], c[2], c[3], c[4], 4 if c[5] is None else c[5], c[6], c[7]) for c in g["cubics"]])
    got = sc.trace(g["rays_in"].copy())
    want = g["intersect_out"]
    rep = compare_hits(want, got)
    assert rep["id_mismatch"] == 0 and rep["hit_miss_disagree"] == 0 and rep["tie"] <= 4, rep
    assert rep["max_rel_t"] <= 1e-4 and rep["max_abs_uv"] <= (5e-3 if rnd else 2e-4) and rep["miss_untouched"], rep
    ok = (got["geomID"] == want["geomID"]) & (got["primID"] == want["primID"]) & (got["geomID"] != 0xFFFFFFFF)
    assert ((want["geomID"] >= 1) & ok).sum() > 1500
    for f in ("Ng_x", "Ng_y", "Ng_z"):
        assert np.allclose(got[f][ok], want[f][ok], rtol=2e-2 if rnd else 1e-3, atol=1e-4 if rnd else 1e-5), f
    occ = sc.trace(rays_of(g["rays_in"]), occluded=True)
    assert (occ["tfar"].view(np.uint32) == g["occluded_out"]["tfar"].view(np.uint32)).all()
    assert np.allclose(sc.bounds(), g["bounds"], rtol=2e-7, atol=0)
    sc.free()


@pytest.mark.parametrize("basis,tess", [("bezier", 4), ("bspline", 9), ("catmull_rom", 16), ("hermite", 1)])
def test_oracle_cubic_curves_vs_reference_live(oracle, basis, tess):
    """Larger randomised check against the reference's outputs: 400 strands of connected cubic curves."""
    from tests.parity import api_trace_mt
    cv, ci, tg = scenes.cubic_hair(400, basis, seed=7)
    v, t = scenes.triangle_sphere(16)
    rng = np.random.RandomState(2)
    org = rng.normal(size=(60000, 3)).astype(np.float32)
    org = org / np.linalg.norm(org, axis=1, keepdims=True) * 2.5
    d = (-org + rng.normal(scale=0.5, size=org.shape)).astype(np.float32)
    rays = sample_rays(make_rayhits(org, d))
    sc = oracle.scene([(v, t, 0, 0xFFFFFFFF)], cubics=[(cv, ci, 1, 0xFFFFFFFF, basis, tess, tg)])
    want = sc.trace(rays.copy(), nthreads=4)

    def run(R):
        dev = R.new_device(None)
        rs = R.rtcNewScene(dev)
        keep = [R.add_triangle_mesh(dev, rs, v, t, mask=0xFFFFFFFF, geom_id=0)[1], R.add_flat_cubic_curves(dev, rs, cv, ci, basis, tess, tg, mask=0xFFFFFFFF, geom_id=1)[1]]
        R.rtcCommitScene(rs)
        R.check(dev)
        out = api_trace_mt(R, rs, rays.copy(), 4), api_trace_mt(R, rs, rays_of(rays), 4, occluded=True), {}
        R.rtcReleaseScene(rs)
        R.rtcReleaseDevice(dev)
        del keep
        return out
    ref, ro, _ = reference_run(f"curves_flat_{basis}", rays, run)
    rep = compare_hits(ref, want)
    # a ray through the very edge of a ribbon quad flips with the rounding of U / V (none at this seed; 4e-6 of the rays of
    # bench.py's fur ball): every difference must be such a graze
    from tests.parity import unexplained_ribbon_disagreements
    n_differ, unexplained = unexplained_ribbon_disagreements(ref, want, {1})
    assert (ref["geomID"] == 1).sum() > len(rays) // 12 and n_differ <= 2 and unexplained == 0 and rep["tie"] <= 4, (rep, n_differ, unexplained)
    assert rep["max_rel_t"] <= 1e-4 and rep["max_abs_uv"] <= 4e-4, rep
    wo = sc.trace(rays_of(rays), occluded=True, nthreads=4)
    assert ((ro["tfar"] < 0) != (wo["tfar"] < 0)).sum() <= 2
    sc.free()


@pytest.mark.parametrize("basis", ["bezier", "bspline", "catmull_rom", "hermite"])
def test_oracle_round_cubic_curves_vs_reference_live(oracle, basis):
    """ROUND cubic curves (sweep intersector) against the reference's outputs: 400 strands.  The hit is the root of a Newton
    iteration, so the two implementations may part where the problem is ill-conditioned -- on the silhouette of the tube; every
    differing ray must be such a graze (tests/parity.py sweep_disagreements; seen: 0-3 of 60 000)."""
    from tests.parity import api_trace_mt, sweep_disagreements
    cv, ci, tg = scenes.cubic_hair(400, basis, seed=8)
    v, t = scenes.triangle_sphere(16)
    rng = np.random.RandomState(10)
    org = rng.normal(size=(60000, 3)).astype(np.float32)
    org = org / np.linalg.norm(org, axis=1, keepdims=True) * 2.5
    d = (-org + rng.normal(scale=0.5, size=org.shape)).astype(np.float32)
    rays = sample_rays(make_rayhits(org, d))
    sc = oracle.scene([(v, t, 0, 0xFFFFFFFF)], cubics=[(cv, ci, 1, 0xFFFFFFFF, basis, 4, tg, True)])
    want = sc.trace(rays.copy(), nthreads=4)

    def run(R):
        dev = R.new_device(None)
        rs = R.rtcNewScene(dev)
        keep = [R.add_triangle_mesh(dev, rs, v, t, mask=0xFFFFFFFF, geom_id=0)[1], R.add_flat_cubic_curves(dev, rs, cv, ci, basis, None, tg, mask=0xFFFFFFFF, geom_id=1, round=True)[1]]
        R.rtcCommitScene(rs)
        R.check(dev)
        out = api_trace_mt(R, rs, rays.copy(), 4), api_trace_mt(R, rs, rays_of(rays), 4, occluded=True), {}
        R.rtcReleaseScene(rs)
        R.rtcReleaseDevice(dev)
        del keep
        return out
    ref, ro, _ = reference_run(f"curves_round_{basis}", rays, run)
    n_differ, unexplained = sweep_disagreements(rays, ref, want, {1})
    assert (ref["geomID"] == 1).sum() > len(rays) // 12 and n_differ <= 8 and unexplained == 0, (n_differ, unexplained)
    wo = sc.trace(rays_of(rays), occluded=True, nthreads=4)
    assert ((ro["tfar"] < 0) != (wo["tfar"] < 0)).sum() <= n_differ
    sc.free()


def test_oracle_points_vs_golden(oracle):
    """Point primitives (sphere_intersector.h, disc_intersector.h) restated in oracle/embree_oracle.c against the reference's own
    outputs: sphere / ray-facing disc / oriented disc sets (geometry masks, an invalid centre, a negative radius, ray origins
    inside spheres) around a triangle sphere."""
    from tests.conftest import load_golden_points
    from tests.parity import point_disagreements
    g = load_golden_points()
    sc = oracle.scene(g["meshes"], points=g["points"])
    got = sc.trace(g["rays_in"].copy())
    want = g["intersect_out"]
    rep = compare_hits(want, got)
    n_differ, unexplained = point_disagreements(g["rays_in"], want, got, {s[3]: (s[0], s[1], s[2]) for s in g["points"]})
    assert n_differ <= 2 and unexplained == 0, (rep, n_differ, unexplained)
    assert all((want["geomID"] == k).sum() > 150 for k in (1, 2, 3)), rep
    assert rep["max_rel_t"] <= 1e-4 and rep["max_abs_uv"] <= 1e-6 and rep["miss_untouched"], rep
    pt = np.isin(got["geomID"], [1, 2, 3])
    assert (got["u"][pt] == 0).all() and (got["v"][pt] == 0).all() and (want["u"][pt] == 0).all()
    ok = (got["geomID"] == want["geomID"]) & (got["primID"] == want["primID"]) & (got["geomID"] != 0xFFFFFFFF)
    for f in ("Ng_x", "Ng_y", "Ng_z"):
        assert np.allclose(got[f][ok], want[f][ok], rtol=1e-3, atol=2e-5), f
    occ = sc.trace(rays_of(g["rays_in"]), occluded=True)
    assert ((occ["tfar"] == -np.inf) != (g["occluded_out"]["tfar"] == -np.inf)).sum() <= n_differ
    assert np.array_equal(sc.bounds(), g["bounds"])
    sc.free()


@pytest.mark.parametrize("kind", ["sphere", "disc", "oriented_disc"])
def test_oracle_points_vs_live_reference(oracle, kind):
    """Rays against 4 000 points of one kind, oracle next to the reference's outputs."""
    from tests.parity import point_disagreements
    rng = np.random.RandomState(5)
    n, m = 4000, 60000
    pv = np.concatenate([rng.uniform(-1, 1, (n, 3)), rng.uniform(0.01, 0.08, (n, 1))], 1).astype(np.float32)
    pn = rng.normal(size=(n, 3)).astype(np.float32)
    org = rng.normal(size=(m, 3)).astype(np.float32)
    org = org / np.linalg.norm(org, axis=1, keepdims=True) * rng.uniform(0.0, 2.5, (m, 1)).astype(np.float32)
    d = ((rng.uniform(-1, 1, (m, 3)) - org) * rng.uniform(0.3, 3, (m, 1))).astype(np.float32)
    rays = make_rayhits(org, d, tnear=1e-3)
    rays["tfar"][::7] = 0.9
    rays = sample_rays(rays)

    def run(R):
        dev = R.new_device(None)
        sc = R.rtcNewScene(dev)
        _, keep = R.add_points(dev, sc, pv, kind, normals=pn, geom_id=3)
        R.rtcCommitScene(sc)
        R.check(dev)
        out = R.intersect(sc, rays.copy(), "1"), R.occluded(sc, rays_of(rays), "1"), {}
        R.rtcReleaseScene(sc)
        R.rtcReleaseDevice(dev)
        return out
    want, wocc, _ = reference_run(f"points_{kind}", rays, run)
    o = oracle.scene([], points=[(pv, kind, pn if kind == "oriented_disc" else None, 3, 0xFFFFFFFF)])
    got = o.trace(rays.copy(), nthreads=8)
    gocc = o.trace(rays_of(rays), occluded=True, nthreads=8)
    rep = compare_hits(want, got, 1e-4)
    n_differ, unexplained = point_disagreements(rays, want, got, {3: (pv, kind, pn)})
    assert rep["hits"] > len(rays) // 6 and n_differ <= 4 and unexplained == 0, (rep, n_differ, unexplained)
    assert rep["max_rel_t"] <= 1e-4 and rep["max_abs_uv"] == 0.0, rep
    assert ((wocc["tfar"] == -np.inf) != (gocc["tfar"] == -np.inf)).sum() <= n_differ
    o.free()


def test_oracle_instanced_curves_and_points_vs_live_reference(oracle):
    """Instances of a scene that holds every curve and point kind (instance_intersector.cpp:15-67 runs the child's curve accel on the
    object-space ray as well): oracle next to the reference's outputs, rays through six instances under rotation, non-uniform
    scale and translation, with instance and geometry masks."""
    from tests.parity import build_instanced_hair, instanced_hair_scene
    S = instanced_hair_scene()
    rays = sample_rays(S["rays"], 1152)

    def run(R):
        from embree_b200.rtc import RTCBounds
        import ctypes as C
        dev = R.new_device(None)
        top, child, keep = build_instanced_hair(R, dev, S)
        out = R.intersect(top, rays.copy(), "1"), R.occluded(top, rays_of(rays), "1")
        b = RTCBounds()
        R.rtcGetSceneBounds(top, C.byref(b))
        R.rtcReleaseScene(top)
        R.rtcReleaseScene(child)
        R.rtcReleaseDevice(dev)
        return out + ({"bounds": np.float32([b.lower_x, b.lower_y, b.lower_z, b.upper_x, b.upper_y, b.upper_z])},)
    want, wocc, extra = reference_run("instanced_curves_points", rays, run)
    oc = oracle.scene([(S["mesh"][0], S["mesh"][1], 0, 0xFFFFFFFF)], curves=S["curves"], cubics=S["cubics"], points=S["points"])
    ot = oracle.scene([], instances=[(oc, m, i, S["masks"][i]) for i, m in enumerate(S["xfms"])])
    got = ot.trace(rays.copy(), nthreads=8)
    gocc = ot.trace(rays_of(rays), occluded=True, nthreads=8)
    rep = compare_hits(want, got, 1e-4)
    per_geom = [int((want["geomID"] == g).sum()) for g in range(8)]
    assert min(per_geom) > 40 * len(rays) // len(S["rays"]) and (want["instID"][want["geomID"] != 0xFFFFFFFF] < len(S["xfms"])).all(), per_geom
    # grazing rays of the curve kinds may flip (see the per-kind tests); nothing systematic
    assert rep["id_mismatch"] + rep["hit_miss_disagree"] <= 6 and rep["max_rel_t"] <= 2e-4, (rep, per_geom)
    same = (want["geomID"] == got["geomID"]) & (want["primID"] == got["primID"]) & (want["geomID"] != 0xFFFFFFFF)
    assert (want["instID"][same] == got["instID"][same]).all()
    assert ((wocc["tfar"] == -np.inf) != (gocc["tfar"] == -np.inf)).sum() <= 6
    assert np.allclose(ot.bounds(), extra["bounds"], rtol=1e-5, atol=1e-5)
    ot.free()
    oc.free()


@pytest.mark.parametrize("kind", ["sphere", "disc", "oriented_disc"])
def test_oracle_point_edge_cases_vs_live_reference(oracle, kind):
    """The corners of the point tests' domain (tests/parity.py point_edge_cases: zero / huge radii, far centres, origins at the centre,
    inside and on the surface, tnear / tfar cutting between front and back hit, |dir| from 1e-3 to 1e3, rays parallel to a disc,
    non-unit normals): oracle next to the reference's outputs; a difference must sit on a decision boundary of the test."""
    from tests.parity import point_disagreements, point_edge_cases
    pv, pn, rays = point_edge_cases()
    n_all = len(rays)
    rays = sample_rays(rays)

    def run(R):
        dev = R.new_device(None)
        sc = R.rtcNewScene(dev)
        _, keep = R.add_points(dev, sc, pv, kind, normals=pn, geom_id=0)
        R.rtcCommitScene(sc)
        R.check(dev)
        out = R.intersect(sc, rays.copy(), "1"), R.occluded(sc, rays_of(rays), "1"), {}
        R.rtcReleaseScene(sc)
        R.rtcReleaseDevice(dev)
        return out
    want, wocc, _ = reference_run(f"point_edge_cases_{kind}", rays, run)
    o = oracle.scene([], points=[(pv, kind, pn if kind == "oriented_disc" else None, 0, 0xFFFFFFFF)])
    got = o.trace(rays.copy())
    gocc = o.trace(rays_of(rays), occluded=True)
    o.free()
    rep = compare_hits(want, got, 1e-4)
    # (t_tol: the same point at different distances counts as a difference as well, measured against the size of the problem in units of t --
    # a hit at t ~ 1e-10 from an origin on the surface has no relative accuracy)
    n_differ, unexplained = point_disagreements(rays, want, got, {0: (pv, kind, pn)}, margin=2e-4, t_tol=1e-4)
    assert rep["hits"] > 1000 * len(rays) // n_all and unexplained == 0 and n_differ <= 0.01 * len(rays), (rep, n_differ, unexplained)
    assert ((wocc["tfar"] == -np.inf) != (gocc["tfar"] == -np.inf)).sum() <= n_differ
