"""Parity helpers shared by the tests, __graft_entry__.smoke() and bench.py's checker leg.

`load_oracle()` returns the CPU restatement (oracle/liboracle.so); `load_reference()` the unmodified reference
built by oracle/build_ref.py (oracle/_ref/libembree4.so.4) or None when it is not present.  Both are CHECKERS: the
product library never sees them."""
import ctypes as C
import os

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_SO = os.path.join(ROOT, "oracle", "liboracle.so")
REF_SO = os.path.join(ROOT, "oracle", "_ref", "libembree4.so.4")


CUBIC_BASES = ["bezier", "bspline", "catmull_rom", "hermite"]
POINT_KINDS = ["sphere", "disc", "oriented_disc"]


class Oracle:
    def __init__(self, path=ORACLE_SO):
        if not os.path.exists(path):
            raise RuntimeError(f"{path} missing: run `make -C oracle`")
        d = C.CDLL(path)
        d.orc_new.restype = C.c_void_p
        d.orc_free.argtypes = [C.c_void_p]
        d.orc_add_mesh.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_uint, C.c_void_p, C.c_size_t, C.c_uint, C.c_uint, C.c_uint]
        d.orc_commit.argtypes = [C.c_void_p]
        d.orc_add_quad_mesh.argtypes = d.orc_add_mesh.argtypes
        d.orc_add_curves.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_uint, C.c_void_p, C.c_size_t, C.c_uint, C.c_void_p, C.c_uint, C.c_uint]
        d.orc_add_curves_typed.argtypes = d.orc_add_curves.argtypes + [C.c_int]
        d.orc_add_cubic_curves.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_uint, C.c_void_p, C.c_size_t, C.c_uint, C.c_uint, C.c_uint,
                                           C.c_int, C.c_int, C.c_void_p, C.c_size_t, C.c_int]
        d.orc_add_instance.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint, C.c_uint]
        d.orc_add_points.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_uint, C.c_void_p, C.c_size_t, C.c_int, C.c_uint, C.c_uint]
        d.orc_set_robust.argtypes = [C.c_void_p, C.c_int]
        d.orc_trace.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_int]
        d.orc_get_bounds.argtypes = [C.c_void_p, C.c_void_p]
        d.orc_get_stats.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        d.orc_count_stats.argtypes = [C.c_void_p, C.c_int]
        d.orc_api_loop.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_size_t, C.c_int, C.c_void_p, C.c_uint, C.c_int]
        self.d = d

    def scene(self, meshes, robust=False, instances=(), curves=(), cubics=(), points=()):
        """meshes: list of (vertices[nv,3] f32, indices[nt,3] u32 (or [nq,4] for a quad mesh), geomID, mask); instances:
        list of (child OracleScene, xfm[12] column-major 3x4, geomID, mask); curves: list of (vertices[nv,4] f32 (xyz,
        radius), first-vertex indices[ns] u32, flags[ns] u8 or None, geomID, mask) round linear curve sets."""
        return OracleScene(self, meshes, robust, instances, curves, cubics, points)

    def trace(self, v, t, rayhits, occluded=False, mask=0xFFFFFFFF, nthreads=1):
        sc = self.scene([(v, t, 0, mask)])
        out = sc.trace(rayhits, occluded, nthreads)
        sc.free()
        return out


class OracleScene:
    def __init__(self, o, meshes, robust=False, instances=(), curves=(), cubics=(), points=()):
        self.o = o
        self.h = o.d.orc_new()
        o.d.orc_set_robust(self.h, 1 if robust else 0)
        self.keep = []
        for (v, t, gid, mask) in meshes:
            v = np.ascontiguousarray(v, np.float32).reshape(-1, 3)
            t = np.ascontiguousarray(t, np.uint32)
            quad = t.ndim == 2 and t.shape[1] == 4
            t = t.reshape(-1, 4 if quad else 3)
            self.keep += [v, t]
            (o.d.orc_add_quad_mesh if quad else o.d.orc_add_mesh)(self.h, v.ctypes.data, 12, v.shape[0], t.ctypes.data,
                                                                   16 if quad else 12, t.shape[0], gid, mask)
        for entry in curves:      # (vertices4, indices, flags or None, geomID, mask[, flat]); flat: RTC_GEOMETRY_TYPE_FLAT_LINEAR_CURVE
            cv, ci, cf, gid, mask = entry[:5]
            flat = len(entry) > 5 and bool(entry[5])
            cv = np.ascontiguousarray(cv, np.float32).reshape(-1, 4)
            ci = np.ascontiguousarray(ci, np.uint32).reshape(-1)
            cf = None if cf is None else np.ascontiguousarray(cf, np.uint8).reshape(-1)
            self.keep += [cv, ci, cf]
            o.d.orc_add_curves_typed(self.h, cv.ctypes.data, 16, cv.shape[0], ci.ctypes.data, 4, ci.shape[0],
                                     None if cf is None else cf.ctypes.data, gid, mask, 1 if flat else 0)
        for entry in cubics:   # cubic curves: basis 'bezier' | 'bspline' | 'catmull_rom' | 'hermite'; 8th element True: ROUND (swept) instead of flat
            cv, ci, gid, mask, basis, tess, tang = entry[:7]
            rnd = len(entry) > 7 and bool(entry[7])
            cv = np.ascontiguousarray(cv, np.float32).reshape(-1, 4)
            ci = np.ascontiguousarray(ci, np.uint32).reshape(-1)
            tg = None if tang is None else np.ascontiguousarray(tang, np.float32).reshape(-1, 4)
            self.keep += [cv, ci, tg]
            o.d.orc_add_cubic_curves(self.h, cv.ctypes.data, 16, cv.shape[0], ci.ctypes.data, 4, ci.shape[0], gid, mask,
                                     CUBIC_BASES.index(basis), int(tess), None if tg is None else tg.ctypes.data, 16, 1 if rnd else 0)
        for (pv, kind, normals, gid, mask) in points:   # point primitives: vertices4 (centre, radius), kind 'sphere' | 'disc' | 'oriented_disc', normals[n,3] or None
            pv = np.ascontiguousarray(pv, np.float32).reshape(-1, 4)
            pn = None if normals is None else np.ascontiguousarray(normals, np.float32).reshape(-1, 3)
            self.keep += [pv, pn]
            o.d.orc_add_points(self.h, pv.ctypes.data, 16, pv.shape[0], None if pn is None else pn.ctypes.data, 12, POINT_KINDS.index(kind), gid, mask)
        for (child, xfm, gid, mask) in instances:
            m = np.ascontiguousarray(xfm, np.float32).reshape(12)
            self.keep += [child, m]
            o.d.orc_add_instance(self.h, child.h, m.ctypes.data, gid, mask)
        o.d.orc_commit(self.h)

    def trace(self, rays, occluded=False, nthreads=1):
        self.o.d.orc_trace(self.h, rays.ctypes.data, len(rays), 1 if occluded else 0, nthreads)
        return rays

    def bounds(self):
        b = np.zeros(6, np.float32)
        self.o.d.orc_get_bounds(self.h, b.ctypes.data)
        return b

    def stats(self):
        s = np.zeros(6, np.uint64)
        sah = C.c_double()
        self.o.d.orc_get_stats(self.h, s.ctypes.data, C.byref(sah))
        return dict(prims=int(s[0]), nodes=int(s[1]), blocks=int(s[2]), trav_nodes=int(s[3]), trav_leaves=int(s[4]),
                    trav_blocks=int(s[5]), sah=sah.value)

    def count_stats(self, on=True):
        self.o.d.orc_count_stats(self.h, 1 if on else 0)

    def free(self):
        if self.h:
            self.o.d.orc_free(self.h)
            self.h = None


_oracle = None


def load_oracle():
    global _oracle
    if _oracle is None:
        _oracle = Oracle()
    return _oracle


_ref = None


def load_reference():
    """The unmodified reference library through the same ctypes binding, or None if oracle/_ref was not built."""
    global _ref
    if _ref is None and os.path.exists(REF_SO):
        from embree_b200.rtc import RTCLib
        _ref = RTCLib(REF_SO)
    return _ref


REFERENCE_RUNS = os.path.join(ROOT, "tests", "golden", "reference_runs")
HIT_FIELDS = ("tfar", "Ng_x", "Ng_y", "Ng_z", "u", "v", "primID", "instID", "instPrimID")


def sample_rays(rays, n=576):
    """A seeded random sample of n rays, in stream order: the rays a reference-run fixture holds outputs for.  (A stride
    would alias with the tests' periodic patterns -- ray masks by index mod 4, tfar on every 7th ray.)"""
    idx = np.sort(np.random.default_rng(0).choice(len(rays), min(n, len(rays)), replace=False))
    return rays[idx].copy()


def reference_run(case, rays, run):
    """The unmodified reference's (rtcIntersect1 records, rtcOccluded1 records, extras) for `rays`, read from
    tests/golden/reference_runs/<case>.npz.  With RTCB200_RECORD_REFERENCE=1 and oracle/_ref built, run(R) computes them
    with the reference library R first and rewrites the fixture (extras: a dict of small arrays, e.g. scene bounds).
    The file keeps geomID for every ray, the other hit fields for the rays that hit, and one occluded bit per ray: a miss
    leaves the RTCRayHit record as it came in, a ray that is not occluded keeps its tfar (checked when recording)."""
    import hashlib
    from embree_b200.rtc import rays_of
    path = os.path.join(REFERENCE_RUNS, case + ".npz")
    digest = np.frombuffer(hashlib.sha256(rays.tobytes()).digest(), np.uint8)
    if os.environ.get("RTCB200_RECORD_REFERENCE"):
        R = load_reference()
        assert R is not None, "RTCB200_RECORD_REFERENCE needs oracle/_ref (python oracle/build_ref.py)"
        hit, occ, extras = run(R)
        h = hit["geomID"] != 0xFFFFFFFF
        o = occ["tfar"] == -np.inf
        assert hit[~h].tobytes() == rays[~h].tobytes(), f"{case}: the reference changed the record of a miss"
        assert occ[~o].tobytes() == rays_of(rays)[~o].tobytes(), f"{case}: the reference changed a ray that is not occluded"
        os.makedirs(REFERENCE_RUNS, exist_ok=True)
        np.savez_compressed(path, rays_sha256=digest, geomID=hit["geomID"], occluded=np.packbits(o),
                            **{f: hit[f][h] for f in HIT_FIELDS}, **{"x_" + k: np.asarray(v) for k, v in extras.items()})
    z = np.load(path)
    assert (z["rays_sha256"] == digest).all(), f"{case}: the test's rays no longer reproduce the rays of the fixture"
    hit, occ = rays.copy(), rays_of(rays)
    hit["geomID"] = z["geomID"]
    h = hit["geomID"] != 0xFFFFFFFF
    for f in HIT_FIELDS:
        hit[f][h] = z[f]
    occ["tfar"][np.unpackbits(z["occluded"], count=len(rays)).astype(bool)] = -np.inf
    return hit, occ, {k[2:]: z[k] for k in z.files if k.startswith("x_")}


def api_trace_mt(lib, scene, recs, nthreads, K=1, occluded=False, coherent=False, valid=None):
    """Loop lib's rtcIntersect1 / rtcOccluded1 / rtcIntersect{K} over `recs` on `nthreads` host threads (FTZ|DAZ set),
    i.e. how a host application drives the reference (BASELINE.md section 4)."""
    name = ("rtcOccluded" if occluded else "rtcIntersect") + str(K)
    fn = C.cast(getattr(lib.dll, name), C.c_void_p)
    o = load_oracle()
    o.d.orc_api_loop(fn, C.c_void_p(scene), recs.ctypes.data, len(recs), recs.dtype.itemsize, K,
                     valid.ctypes.data if valid is not None else None, (1 << 16) if coherent else 0, nthreads)
    return recs


TIE_ULPS = 4


def _share_a_vertex(meshes, ga, pa, gb, pb):
    """Per pair of (geomID, primID): do the two triangles have a vertex POSITION in common (shared edge / vertex)?"""
    by_id = {int(gid): (np.asarray(v, np.float32), np.asarray(t)) for (v, t, gid, _m) in meshes}
    out = np.zeros(len(ga), bool)
    for i in range(len(ga)):
        va, ta = by_id[int(ga[i])]
        vb, tb = by_id[int(gb[i])]
        if ta.shape[1] != 3 or tb.shape[1] != 3:
            out[i] = True          # quads: the two halves of one quad share the diagonal by construction
            continue
        A, B = va[ta[int(pa[i])]], vb[tb[int(pb[i])]]
        out[i] = bool((A[:, None, :] == B[None, :, :]).all(axis=2).any())
    return out


def compare_hits(want, got, tol=1e-4, meshes=None):
    """Hit-record parity as BASELINE.json states it: primID/geomID/instID exact, tfar/u/v within `tol` relative
    (u, v relative to 1 since they live in [0,1]).  Returns counts.  `tie` = id mismatches where both libraries report
    the SAME distance -- tfar within TIE_ULPS ulp (the reference's rcp+Newton vs IEEE division is 1 ulp) -- and, when
    `meshes` = [(verts, tris, geomID, mask), ...] is given, the two primitives share a vertex position: the ray hits
    exactly on a shared edge / vertex, both triangles accept it at the same t, and the reference's own winner depends on
    its traversal order (SURVEY 7 hard part 2).  Every other id difference is `id_mismatch`."""
    n = len(want)
    wh = want["geomID"] != 0xFFFFFFFF
    gh = got["geomID"] != 0xFFFFFFFF
    both = wh & gh
    id_mis = both & ((want["primID"] != got["primID"]) | (want["geomID"] != got["geomID"]) | (want["instID"] != got["instID"]))
    wt, gt = want["tfar"].astype(np.float64), got["tfar"].astype(np.float64)
    with np.errstate(invalid="ignore", divide="ignore"):
        rel_t = np.where(both, np.abs(wt - gt) / np.maximum(np.abs(wt), 1e-30), 0.0)
    ulps = np.abs(want["tfar"].view(np.int32).astype(np.int64) - got["tfar"].view(np.int32).astype(np.int64))
    same_t = both & (ulps <= TIE_ULPS) & (want["tfar"] > 0) & (got["tfar"] > 0)
    tie = id_mis & same_t
    shared_checked = meshes is not None
    if shared_checked and tie.any():
        k = np.nonzero(tie)[0]
        tie[k] = _share_a_vertex(meshes, want["geomID"][k], want["primID"][k], got["geomID"][k], got["primID"][k])
    hard = id_mis & ~tie
    ok = both & ~id_mis
    du = np.abs(want["u"].astype(np.float64) - got["u"])[ok]
    dv = np.abs(want["v"].astype(np.float64) - got["v"])[ok]
    ng_exact = all(((want[f].view(np.uint32) == got[f].view(np.uint32)) | ~ok).all() for f in ("Ng_x", "Ng_y", "Ng_z"))
    miss_tfar_same = ((want["tfar"].view(np.uint32) == got["tfar"].view(np.uint32)) | wh | gh).all()
    return dict(n=int(n), hits=int(wh.sum()), id_mismatch=int(hard.sum()), tie=int(tie.sum()),
                tie_rule=f"tfar within {TIE_ULPS} ulp" + (" and a shared vertex" if shared_checked else ""),
                hit_miss_disagree=int((wh != gh).sum()),
                max_rel_t=float(rel_t[ok].max()) if ok.any() else 0.0,
                max_abs_uv=float(max(du.max() if du.size else 0.0, dv.max() if dv.size else 0.0)),
                ng_bit_exact=bool(ng_exact), miss_untouched=bool(miss_tfar_same))


def explain_hit_miss(oracle, rays, want, got, single_prim_scene):
    """Every ray on which `got` (the GPU) and `want` (the oracle / the reference) disagree about hit vs miss must be an
    edge case of the REFERENCE algorithm, shown ray by ray -- none is waved through:
      * want hits, got misses: never acceptable (returned in `lost`);
      * got hits, want misses: `single_prim_scene(geomID, primID, instID)` builds an oracle scene that holds ONLY the
        primitive the GPU reports; the reference's own triangle arithmetic must accept it there with bit-equal t, u, v.
        Then the full-scene miss is the reference's non-conservative fast box test culling that leaf by a rounding error
        (node_intersector1.h:484-531 carries no padding; ours is padded by 2 ulp), not a wrong GPU hit.
    Returns (lost, unexplained_extra)."""
    wh = want["geomID"] != 0xFFFFFFFF
    gh = got["geomID"] != 0xFFFFFFFF
    lost = int((wh & ~gh).sum())
    bad = 0
    for i in np.nonzero(gh & ~wh)[0]:
        sc = single_prim_scene(int(got["geomID"][i]), int(got["primID"][i]), int(got["instID"][i]))
        r = rays[i:i + 1].copy()
        sc.trace(r)
        same = all(r[f].view(np.uint32)[0] == got[f].view(np.uint32)[i] for f in ("tfar", "u", "v"))
        bad += 0 if (r["geomID"][0] != 0xFFFFFFFF and same) else 1
        sc.free()
    return lost, bad


def curve_grazing(cv, ci, prim, ray, limit=1e-2):
    """Is `ray` (one RTCRayHit record) near-tangent to round linear segment `prim`?  The cone hit exists iff the
    discriminant D = B^2 - 4AC of roundline_intersector.h:296-325 is >= 0; B and C are differences of nearly equal
    products, so when D is a small fraction of B^2 (evaluated here in float64) its fp32 sign depends on the order of
    rounding / FMA contraction, which differs between the reference's AVX code and any other implementation.  Also true
    for the end spheres (h2 of :356, :380 against O1dO^2)."""
    vid = int(ci[prim])
    v0, v1 = cv[vid].astype(np.float64), cv[vid + 1].astype(np.float64)
    O = np.array([ray["org_x"], ray["org_y"], ray["org_z"]], np.float64)
    D = np.array([ray["dir_x"], ray["dir_y"], ray["dir_z"]], np.float64)
    dP, dr = v1[:3] - v0[:3], v1[3] - v0[3]
    g = dP @ dP - dr * dr
    org = O + (((0.5 * (v0[:3] + v1[:3]) - O) @ D) / (D @ D)) * D
    Ov = org - v0[:3]
    dOdP, OdP = dP @ D, dP @ Ov
    yp = OdP + v0[3] * dr
    A, B = g * (D @ D) - dOdP ** 2, 2 * (g * (D @ Ov) - dOdP * yp)
    Cc = g * (Ov @ Ov) - OdP ** 2 - v0[3] ** 2 * (dP @ dP) - 2 * v0[3] * dr * OdP
    graz = abs(B * B - 4 * A * Cc) <= limit * max(B * B, abs(4 * A * Cc))
    for c, r in ((v0, v0[3]), (v1, v1[3])):
        O1 = org - c[:3]
        b1 = O1 @ D
        h2 = b1 * b1 - (D @ D) * (O1 @ O1 - r * r)
        graz = graz or abs(h2) <= limit * max(b1 * b1, (D @ D) * abs(O1 @ O1 - r * r))
    return bool(graz)


def unexplained_curve_disagreements(rays, a, b, curve_sets):
    """Rays on which two implementations of the curve test disagree (hit vs miss, or different primitives at different
    distances) and for which NO involved curve segment is near-tangent to the ray (curve_grazing).  curve_sets:
    {geomID: (vertices[nv,4], first-vertex indices)}.  Ties (same distance within TIE_ULPS) are not disagreements."""
    ah, bh = a["geomID"] != 0xFFFFFFFF, b["geomID"] != 0xFFFFFFFF
    ulps = np.abs(a["tfar"].view(np.int32).astype(np.int64) - b["tfar"].view(np.int32).astype(np.int64))
    differ = (ah != bh) | (ah & bh & ((a["primID"] != b["primID"]) | (a["geomID"] != b["geomID"])) & (ulps > TIE_ULPS))
    bad = 0
    for i in np.nonzero(differ)[0]:
        involved = [(int(x["geomID"][i]), int(x["primID"][i])) for x in (a, b) if int(x["geomID"][i]) in curve_sets]
        if not any(curve_grazing(curve_sets[g][0], curve_sets[g][1], p, rays[i]) for (g, p) in involved):
            bad += 1
    return int(differ.sum()), bad


def unexplained_ribbon_disagreements(a, b, curve_geoms, vmin=0.999):
    """Flat cubic curves: rays on which two implementations of the ribbon test disagree (hit vs miss, or different curves
    at different distances), and how many of them are NOT explained by a graze: the nearer of the two hits must lie on the
    very edge of its ribbon (|v| >= vmin; v runs from -1 to 1 across the ribbon), where the sign of the quad's edge
    functions U, V (quad_intersector.h:52-56) is decided by rounding -- the reference evaluates them with approximate
    reciprocal square roots, this library with exact ones.  Returns (differing rays, unexplained ones)."""
    ah, bh = a["geomID"] != 0xFFFFFFFF, b["geomID"] != 0xFFFFFFFF
    ulps = np.abs(a["tfar"].view(np.int32).astype(np.int64) - b["tfar"].view(np.int32).astype(np.int64))
    differ = (ah != bh) | (ah & bh & ((a["primID"] != b["primID"]) | (a["geomID"] != b["geomID"])) & (ulps > TIE_ULPS))
    bad = 0
    for i in np.nonzero(differ)[0]:
        cands = [x for x, h in ((a, ah[i]), (b, bh[i])) if h]
        near = min(cands, key=lambda x: float(x["tfar"][i]))
        if not (int(near["geomID"][i]) in curve_geoms and abs(float(near["v"][i])) >= vmin):
            bad += 1
    return int(differ.sum()), bad


def sweep_disagreements(rays, a, b, curve_geoms, tol=1e-4, cos_max=0.1):
    """Round (swept) cubic curves: the hit is the result of a Newton iteration started from bounding-cylinder estimates
    (curve_intersector_sweep.h:59-140), so two implementations can converge to different roots, or one of them not at all,
    where the problem is ill-conditioned: on the silhouette of the tube, where the ray is tangent to the surface.  Returns
    (differing rays, unexplained ones): a ray differs when hit / miss, the curve or the distance (beyond `tol` relative)
    differ; it is explained when the nearer of the two hits is a curve hit whose normal is perpendicular to the ray
    (|cos(Ng, dir)| < cos_max)."""
    ah, bh = a["geomID"] != 0xFFFFFFFF, b["geomID"] != 0xFFFFFFFF
    with np.errstate(invalid="ignore", divide="ignore"):
        rel = np.abs(a["tfar"] - b["tfar"]) / np.maximum(np.abs(a["tfar"]), 1e-30)
    ulps = np.abs(a["tfar"].view(np.int32).astype(np.int64) - b["tfar"].view(np.int32).astype(np.int64))
    # (two curves that meet at a joint and are hit at the same distance are a tie, not a difference)
    differ = (ah != bh) | (ah & bh & ((((a["primID"] != b["primID"]) | (a["geomID"] != b["geomID"])) & (ulps > TIE_ULPS)) | (rel > tol)))
    bad = 0
    for i in np.nonzero(differ)[0]:
        cands = [x for x, h in ((a, ah[i]), (b, bh[i])) if h]
        near = min(cands, key=lambda x: float(x["tfar"][i]))
        ng = np.array([near["Ng_x"][i], near["Ng_y"][i], near["Ng_z"][i]], np.float64)
        d = np.array([rays["dir_x"][i], rays["dir_y"][i], rays["dir_z"][i]], np.float64)
        c = abs(ng @ d) / max(np.linalg.norm(ng) * np.linalg.norm(d), 1e-300)
        if not (int(near["geomID"][i]) in curve_geoms and c < cos_max):
            bad += 1
    return int(differ.sum()), bad


def point_disagreements(rays, a, b, point_sets, margin=1e-4, t_tol=None):
    """Point primitives: rays on which two implementations disagree (hit vs miss, or different primitives at different
    distances), and how many of them are NOT explained by a graze.  point_sets: {geomID: (vertices[n,4], kind, normals or None)}.
    A disagreement is explained when, for a point one side reports and the other does not, the exact (float64) test sits on a
    decision boundary within `margin` relative: the ray is tangent to the sphere / passes through the rim of the disc, or the hit
    distance coincides with tnear / tfar (the reference evaluates 1 / dir^2 with a refined hardware approximation, this library
    with the exact reciprocal).  `t_tol`: also count the same point reported at distances that differ by more than t_tol relative to the
    size of the problem in units of t (front hit on one side, back hit on the other).  Returns (differing rays, unexplained ones)."""
    ah, bh = a["geomID"] != 0xFFFFFFFF, b["geomID"] != 0xFFFFFFFF
    ulps = np.abs(a["tfar"].view(np.int32).astype(np.int64) - b["tfar"].view(np.int32).astype(np.int64))
    differ = (ah != bh) | (ah & bh & ((a["primID"] != b["primID"]) | (a["geomID"] != b["geomID"])) & (ulps > TIE_ULPS))
    if t_tol is not None:   # the same point at different distances (front hit on one side, back hit on the other) is a difference too
        k = np.nonzero(ah & bh & (a["primID"] == b["primID"]) & (a["geomID"] == b["geomID"]) & np.isin(a["geomID"], list(point_sets)))[0]
        for g in point_sets:
            kg = k[a["geomID"][k] == g]
            pvg = point_sets[g][0]
            o3 = np.stack([rays["org_x"][kg], rays["org_y"][kg], rays["org_z"][kg]], 1).astype(np.float64)
            d3 = np.stack([rays["dir_x"][kg], rays["dir_y"][kg], rays["dir_z"][kg]], 1).astype(np.float64)
            c3, r3 = pvg[a["primID"][kg], :3].astype(np.float64), pvg[a["primID"][kg], 3].astype(np.float64)
            tscale = (np.linalg.norm(c3 - o3, axis=1) + r3) / np.maximum(np.linalg.norm(d3, axis=1), 1e-30)
            err = np.abs(a["tfar"][kg].astype(np.float64) - b["tfar"][kg]) / np.maximum(np.maximum(np.abs(a["tfar"][kg]), tscale), 1e-30)
            differ[kg[err > t_tol]] = True
    bad = 0
    for i in np.nonzero(differ)[0]:
        o = np.array([rays["org_x"][i], rays["org_y"][i], rays["org_z"][i]], np.float64)
        d = np.array([rays["dir_x"][i], rays["dir_y"][i], rays["dir_z"][i]], np.float64)
        tn, tf = float(rays["tnear"][i]), float(rays["tfar"][i])
        explained = False
        for x, h in ((a, ah[i]), (b, bh[i])):
            g = int(x["geomID"][i])
            if not h or g not in point_sets:
                continue
            pv, kind, pn = point_sets[g]
            c, r = pv[int(x["primID"][i]), :3].astype(np.float64), float(pv[int(x["primID"][i]), 3])
            c0 = c - o
            if kind == "oriented_disc":
                n = pn[int(x["primID"][i])].astype(np.float64)
                t = float(c0 @ n) / float(d @ n)
                ts = [t]
                rim = abs(np.linalg.norm(o + t * d - c) - r) / max(r, 1e-30)
            else:
                proj = float(c0 @ d) / float(d @ d)
                l = np.linalg.norm(c0 - proj * d)
                rim = abs(l - r) / max(r, 1e-30)
                td = np.sqrt(max(r * r - l * l, 0.0) / float(d @ d))
                ts = [proj] if kind == "disc" else [proj - td, proj + td]
            tscale = (np.linalg.norm(c0) + r) / max(np.linalg.norm(d), 1e-30)      # the size of the problem in units of t: a hit at t ~ 0 with tnear = 0 is a boundary case too
            edge = min(min(abs(t - tn), abs(t - tf) if np.isfinite(tf) else np.inf) / max(abs(t), tscale, 1e-30) for t in ts)
            explained |= (rim < margin) or (edge < margin)
        bad += 0 if explained else 1
    return int(differ.sum()), bad


def instanced_hair_scene(seed=3, n_inst=6):
    """A child scene of every curve / point kind around a triangle sphere + `n_inst` instances of it under random affine transforms
    (rotation x non-uniform scale + translation) with instance masks, and rays through the lot.  Returns dict(mesh, curves, cubics,
    points, xfms, masks, rays) in the formats OracleScene / the rtc.py helpers take."""
    from embree_b200 import scenes
    from embree_b200.rtc import make_rayhits
    rng = np.random.RandomState(seed)
    v, t = scenes.triangle_sphere(10)
    v = (v * np.float32(0.5)).astype(np.float32)
    cv, ci, _ = scenes.hair_ball(150, 4, seed=seed + 1, radius=0.5, length=0.5, width=0.03)
    bv, bi, _tg = scenes.cubic_hair(120, "bezier", knots=7, seed=seed + 2, radius=0.5, step=0.08, width=0.02)
    cv2, ci2, _ = scenes.hair_ball(150, 4, seed=seed + 5, radius=0.5, length=0.5, width=0.03)
    bv2, bi2, _tg2 = scenes.cubic_hair(120, "bezier", knots=7, seed=seed + 6, radius=0.5, step=0.08, width=0.02)
    def cloud():
        pc = rng.normal(size=(300, 3)).astype(np.float32)
        pc = pc / np.linalg.norm(pc, axis=1, keepdims=True) * rng.uniform(0.6, 1.1, (300, 1)).astype(np.float32)
        return np.concatenate([pc, rng.uniform(0.02, 0.07, (300, 1)).astype(np.float32)], 1).astype(np.float32)
    pv, pv2, pv3 = cloud(), cloud(), cloud()
    pn = rng.normal(size=(300, 3)).astype(np.float32)
    xfms, masks = [], []
    for i in range(n_inst):
        q, _r = np.linalg.qr(rng.normal(size=(3, 3)))
        m = (q * rng.uniform(0.6, 1.4, 3)[None, :]).astype(np.float32)            # columns vx | vy | vz
        p = (rng.uniform(-2.5, 2.5, 3)).astype(np.float32)
        xfms.append(np.concatenate([m[:, 0], m[:, 1], m[:, 2], p]).astype(np.float32))
        masks.append([0xFFFFFFFF, 0x1, 0x2, 0xFFFFFFFF, 0x3, 0xFFFFFFFF][i % 6])
    m = 30000
    org = rng.uniform(-4, 4, (m, 3)).astype(np.float32)
    tgt = np.stack([x[9:12] for x in xfms])[rng.randint(0, n_inst, m)] + rng.normal(scale=0.5, size=(m, 3)).astype(np.float32)
    d = ((tgt - org) * rng.uniform(0.3, 2.0, (m, 1))).astype(np.float32)
    rays = make_rayhits(org, d)
    rays["mask"][1::3] = 0x1
    rays["mask"][2::3] = 0x2
    rays["tfar"][::9] = 1.0
    return dict(mesh=(v, t), curves=[(cv, ci, None, 1, 0xFFFFFFFF, False), (cv2, ci2, None, 2, 0x5, True)],
                cubics=[(bv, bi, 3, 0xFFFFFFFF, "bezier", 4, None, False), (bv2, bi2, 4, 0xFFFFFFFF, "bezier", 4, None, True)],
                points=[(pv, "sphere", None, 5, 0xFFFFFFFF), (pv2, "disc", None, 6, 0x6), (pv3, "oriented_disc", pn, 7, 0xFFFFFFFF)],
                xfms=xfms, masks=masks, rays=rays)


def build_instanced_hair(L, d, S):
    """The scene of instanced_hair_scene() on a library behind the rtc.py binding: returns (top scene, child scene, keep-alive list)."""
    child = L.rtcNewScene(d)
    keep = [L.add_triangle_mesh(d, child, S["mesh"][0], S["mesh"][1], mask=0xFFFFFFFF, geom_id=0)[1]]
    for (cv, ci, cf, gid, mask, flat) in S["curves"]:
        keep.append(L.add_round_linear_curves(d, child, cv, ci, cf, mask=mask, geom_id=gid, flat=flat)[1])
    for (bv, bi, gid, mask, basis, tess, tang, rnd) in S["cubics"]:
        keep.append(L.add_flat_cubic_curves(d, child, bv, bi, basis, tess, tang, mask=mask, geom_id=gid, round=rnd)[1])
    for (pv, kind, pn, gid, mask) in S["points"]:
        keep.append(L.add_points(d, child, pv, kind, normals=pn if pn is not None else None, mask=mask, geom_id=gid)[1])
    L.rtcCommitScene(child)
    L.check(d)
    top = L.rtcNewScene(d)
    for i, m in enumerate(S["xfms"]):
        L.add_instance(d, top, child, m, mask=S["masks"][i], geom_id=i)
    L.rtcCommitScene(top)
    L.check(d)
    return top, child, keep


def point_edge_cases(seed=77):
    """Point primitives and rays at the corners of the test's domain: zero and large radii, far-away centres, ray origins at the centre /
    inside / on the surface, tnear / tfar windows that cut between the front and the back hit, direction lengths from 1e-3 to 1e3,
    rays parallel to an oriented disc, non-unit normals.  Returns (vertices4, normals, rays)."""
    from embree_b200.rtc import make_rayhits
    rng = np.random.RandomState(seed)
    n = 96
    c = rng.uniform(-1, 1, (n, 3)).astype(np.float32)
    c[::8] *= np.float32(3000.0)                                   # far from the origin
    r = rng.uniform(0.05, 0.3, n).astype(np.float32)
    r[1::8] = 0.0                                                  # degenerate but valid (radius >= 0)
    r[2::8] = 2.5                                                  # contains many ray origins
    r[::8] *= np.float32(300.0)
    pv = np.concatenate([c, r[:, None]], 1).astype(np.float32)
    pn = (rng.normal(size=(n, 3)) * rng.uniform(0.1, 10.0, (n, 1))).astype(np.float32)
    org, d, tn, tf = [], [], [], []
    for i in range(n):
        for k in range(40):
            ci, ri = pv[i, :3].astype(np.float64), max(float(pv[i, 3]), 1e-3)
            u = rng.normal(size=3)
            u /= np.linalg.norm(u)
            mode = k % 8
            if mode == 0:      # from outside, through the point with some offset
                o = ci + u * ri * rng.uniform(1.5, 6.0)
                t = ci + rng.normal(size=3) * ri * 0.7 - o
            elif mode == 1:    # origin at the centre
                o, t = ci.copy(), u
            elif mode == 2:    # origin inside
                o = ci + u * ri * rng.uniform(0.0, 0.95)
                t = rng.normal(size=3)
            elif mode == 3:    # origin (nearly) on the surface, pointing in or out
                o = ci + u * ri
                t = -u + rng.normal(size=3) * 0.8
            elif mode == 4:    # grazing
                w = np.cross(u, rng.normal(size=3))
                w /= np.linalg.norm(w)
                o = ci + u * ri * rng.uniform(0.98, 1.02) - w * ri * 4.0
                t = w
            elif mode == 5:    # parallel to the oriented disc's plane
                nn = pn[i].astype(np.float64)
                w = np.cross(nn, rng.normal(size=3))
                o = ci - w / np.linalg.norm(w) * ri * 3.0 + nn / np.linalg.norm(nn) * ri * rng.uniform(-0.2, 0.2)
                t = w
            else:
                o = rng.uniform(-1.5, 1.5, 3)
                t = ci - o + rng.normal(size=3) * ri
            t = t / max(np.linalg.norm(t), 1e-30) * (10.0 ** rng.uniform(-3, 3))
            org.append(o); d.append(t)
            dist = np.linalg.norm(ci - o) / np.linalg.norm(t)
            tn.append(0.0 if k % 3 else dist * rng.uniform(0.5, 1.2))
            tf.append(np.inf if k % 5 else dist * rng.uniform(0.8, 1.5))
    rays = make_rayhits(np.array(org, np.float32), np.array(d, np.float32))
    rays["tnear"] = np.array(tn, np.float32)
    rays["tfar"] = np.maximum(np.array(tf, np.float32), rays["tnear"])
    return pv, pn, rays
